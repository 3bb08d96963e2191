"""CPU: the host half of collation (collator.pack_host) and its DataLoader-worker stream — no GPU, no libmobgt calls."""
import numpy as np
import torch

from mobgt_b200 import collator, synth


def _case(B=7, cap=20):
    world = synth.make_world("tiny", seed=1)
    return synth.make_items(world, B, cap, seed=3, cfg_id=2)


def _field(hp, name):
    off, shape, dts, nbytes = hp.layout[name]
    return hp.buf[off:off + nbytes].view(np.dtype(dts)).reshape(shape)


def test_pack_host_matches_per_item_loop():
    items = _case()
    hp = collator.pack_host(items)
    ns = np.array([len(np.asarray(it.x)) for it in items])
    assert hp.B == len(items) and hp.N == ns.max() and hp.cells == int((ns.astype(np.int64) ** 2).sum())
    sq = np.concatenate([[0], np.cumsum(ns.astype(np.int64) ** 2)])
    no = np.concatenate([[0], np.cumsum(ns)])
    feat, indeg, outdeg = np.zeros(hp.cells, np.uint8), np.zeros(no[-1], np.int32), np.zeros(no[-1], np.int32)
    for g, it in enumerate(items):                      # wrapper.py:42-53, 97-98 per item
        ei, ea, n = np.asarray(it.edge_index), np.asarray(it.edge_attr).reshape(-1), ns[g]
        feat[sq[g] + ei[0] * n + ei[1]] = ea + 2
        indeg[no[g]:no[g + 1]] = np.bincount(ei[0], minlength=n)
        outdeg[no[g]:no[g + 1]] = np.bincount(ei[1], minlength=n)
    assert np.array_equal(_field(hp, "feat8"), feat)
    assert np.array_equal(_field(hp, "in_deg"), indeg + 1) and np.array_equal(_field(hp, "out_deg"), outdeg + 1)
    assert np.array_equal(_field(hp, "n"), ns) and np.array_equal(_field(hp, "sq_off"), sq)
    assert np.array_equal(_field(hp, "x_nodes"), np.concatenate([np.asarray(it.x).reshape(-1) for it in items]))
    tok_off = _field(hp, "tok_off")
    assert np.array_equal(tok_off, no + np.arange(len(items) + 1))
    tok_pos, rows = _field(hp, "tok_pos"), _field(hp, "node_rows")
    assert (tok_pos[tok_off[:-1]] == 0).all() and (tok_pos[rows] > 0).all() and len(rows) == no[-1]
    for off, shape, dts, nbytes in hp.layout.values():  # every segment 16-byte aligned (typed device views)
        assert off % 16 == 0


def test_worker_stream_shards_batches_in_order():
    a, b = _case(4, 10), _case(6, 16)
    ref = [collator.pack_host(x) for x in (a, b, a, b, a)]
    ds = collator._PackStream([a, b, a, b, a], 512)
    dl = torch.utils.data.DataLoader(ds, batch_size=None, num_workers=2, prefetch_factor=2)
    got = list(dl)
    assert len(got) == 5
    for d, hp in zip(got, ref):
        assert np.array_equal(d["buf"].numpy(), hp.buf) and d["B"] == hp.B and d["cells"] == hp.cells
        assert {k: tuple(v) if not isinstance(v, tuple) else v for k, v in d["layout"].items()}.keys() == hp.layout.keys()


def test_packed_loader_protocol_without_cuda():
    """PackedLoader's one-batch-ahead protocol (current / advance / iteration, end of stream) with a host-only collate_fn and
    no side stream (a side-stream batch must be an object that carries its ready event), so it runs alike with or without CUDA."""
    from mobgt_b200 import collator
    batches = [[i, i + 1] for i in range(5)]
    seen = []
    loader = collator.PackedLoader(iter(batches), collate_fn=lambda items: {"items": list(items)}, num_workers=0, side_stream=False)
    assert loader.current()["items"] == [0, 1]
    loader.advance()
    assert loader.current()["items"] == [1, 2]
    for b in loader:                      # iteration continues from the current batch and advances by itself
        seen.append(b["items"][0])
    assert seen == [1, 2, 3, 4]
    assert loader.current() is None       # end of stream


def test_host_sort_plans_equal_the_device_recipe():
    """pack_host ships the K4-backward sort plans and the attention launch order: they equal what Batch1.build_plans computes
    on the device (ops.sort_plan = torch.sort(stable=True) of the same key streams; stable sorts are unique), for a plain and a
    bucketed (padded) batch."""
    for bucket in (False, True):
        hp = collator.pack_host(_case(B=9, cap=40), bucket=bucket)
        tok_pos, rows = torch.from_numpy(_field(hp, "tok_pos").copy()), torch.from_numpy(_field(hp, "node_rows").copy())
        ind = torch.zeros_like(tok_pos)
        ind[rows] = torch.from_numpy(_field(hp, "in_deg").copy())
        outd = torch.zeros_like(tok_pos)
        outd[rows] = torch.from_numpy(_field(hp, "out_deg").copy())
        keys = {"poi": torch.from_numpy(_field(hp, "x_nodes").copy()).long() - 1, "slot": torch.from_numpy(_field(hp, "slot").copy()),
                "pos": tok_pos, "ind": ind, "outd": outd}
        for name, k in keys.items():
            ks, perm = torch.sort(k.long(), stable=True)
            assert np.array_equal(_field(hp, f"plan_{name}_perm"), perm.int().numpy()), (bucket, name)
            assert np.array_equal(_field(hp, f"plan_{name}_keys"), ks.int().numpy()), (bucket, name)
        n = torch.from_numpy(_field(hp, "n").copy())
        assert np.array_equal(_field(hp, "size_order"), torch.argsort(n, descending=True, stable=True).int().numpy())
