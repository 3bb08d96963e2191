"""Collation: raw dataset items -> `Batch1`, the reference's batch type (collator.py:149-215), B200-first.

The reference's POI collators (collator_foursquare / _gowalla / _toyota, collator.py:310-748) run Floyd-Warshall and
the path walk per item on the CPU, pad everything to the batch maximum as int64, and loop over node pairs in
Python.  Here the host only packs the raw edge lists; the per-pair work runs on the GPU through libmobgt
(K1 + poi_pos), and the batch keeps COMPACT PACKED device tensors (i16 / u8, no padding).  Every reference field
name (`rel_pos` (= `spatial_pos`), `edge_input`, `attn_bias`, `attn_edge_type`, `in_degree`, `out_degree`, `x`, `y`,
`adj`, `adj1`, `time`, `time_normal`, `user`, `cat`, `poi_pos`, `idx`) is still available: it is materialised on
first access with the reference's dtype, shape, "+1" shifts and -inf padding columns (SURVEY.md §8a A1e).
`feature_matrix` (the Laplacian eigenvectors of collator.py:394-410) is never read by the reference forward and
is not produced (None).
"""
import numpy as np
import torch

from . import _C
from .algos import apsp_edge_input_packed, hop_stride


def _to_np(a, dtype=None):
    if isinstance(a, torch.Tensor):
        a = a.cpu().numpy()
    a = np.asarray(a)
    return a.astype(dtype) if dtype is not None else a


class _Staging:
    """Two pinned host buffers used in turn: a buffer is reused only after the copy that read it has completed."""

    def __init__(self):
        self.slots = [None, None]
        self.events = [None, None]
        self.turn = 0

    def get(self, nbytes):
        i = self.turn
        self.turn ^= 1
        if self.events[i] is not None:
            self.events[i].synchronize()
        if self.slots[i] is None or self.slots[i].numel() < nbytes:
            self.slots[i] = torch.empty(max(nbytes, 1 << 20), dtype=torch.uint8).pin_memory()
        return i, self.slots[i]

    def mark(self, i):
        self.events[i] = torch.cuda.Event()
        self.events[i].record()


_staging = {}


class _PackStream(torch.utils.data.IterableDataset):
    """Worker-side half of PackedLoader: worker w packs the batches i = w (mod num_workers) of the stream."""

    def __init__(self, batches, max_node, bucket=False, large_graphs=False):
        self.batches, self.max_node, self.bucket, self.large_graphs = batches, max_node, bucket, large_graphs

    def __iter__(self):
        info = torch.utils.data.get_worker_info()
        w, nw = (info.id, info.num_workers) if info is not None else (0, 1)
        for i, items in enumerate(self.batches):
            if i % nw == w:
                hp = pack_host(items, self.max_node, bucket=self.bucket, large_graphs=self.large_graphs)
                yield dict(buf=torch.from_numpy(hp.buf), layout=hp.layout, B=hp.B, N=hp.N, ns=torch.from_numpy(hp.ns), cells=hp.cells,
                           padded=hp.padded)


class PackedLoader:
    """One-batch-ahead collation (the role of the reference's DataLoader workers, data.py:255-267).  `batches` is an iterable
    of item lists.
      * num_workers = 0: `advance()` packs the next batch on the calling thread — right after the kernels of the current step
        have been enqueued, so the packing, H2D copy and K1 / poi_pos kernels overlap the step's GPU time;
      * num_workers > 0: the numpy packing (`pack_host`) runs in DataLoader worker processes which hand over ONE byte buffer
        per batch through shared memory; the calling thread copies it into the pinned staging buffer and issues the H2D copy
        and the collation kernels (`collate_from_host`).
    side_stream=True (default): the H2D copy and the collation kernels (K1, poi_pos, the K4 sort plans) of batch i+1 are issued
    on a second CUDA stream, so they run concurrently with the kernels of training step i instead of queueing behind them;
    `current()` makes the consumer's stream wait for the batch (event) and registers the batch's memory with that stream.
    """

    def __init__(self, batches, collate_fn=None, num_workers=0, max_node=512, side_stream=True, bucket=False, large_graphs=False,
                 **collate_kw):
        """bucket=True: every batch is padded to a few size buckets (see `pack_host`), so that batches of different graphs
        share packed shapes and the trainer's CUDA graphs replay instead of re-capturing / running eagerly.
        large_graphs=True: graphs of up to MAX_MODEL_NODES (1024) nodes are collated (see `collate_from_host`)."""
        self._kw = dict(collate_kw, large_graphs=large_graphs)
        self._stream = torch.cuda.Stream() if (side_stream and torch.cuda.is_available()) else None
        self._gate = None
        if num_workers > 0:
            ds = _PackStream(batches, max_node, bucket, large_graphs)
            dl = torch.utils.data.DataLoader(ds, batch_size=None, num_workers=num_workers, pin_memory=False, prefetch_factor=2,
                                             persistent_workers=False)
            self._it = iter(dl)
            self._collate = lambda d: collate_from_host(HostPack(d["buf"], d["layout"], d["B"], d["N"], d["ns"], d["cells"], d["padded"]),
                                                        **self._kw)
        else:
            self._it = iter(batches)
            self._collate = collate_fn if collate_fn is not None else (
                lambda items: collate_packed(items, max_node=max_node, bucket=bucket, **self._kw))
        self._next = self._pull()

    def _pull(self):
        try:
            nxt = next(self._it)
        except StopIteration:
            return None
        if self._stream is None:
            return self._collate(nxt)
        if self._gate is not None:
            # start only after everything the consumer had enqueued when it fetched the current batch (the previous step incl.
            # its gradient all-reduce and optimizer): the collation then overlaps the head of the running step, not NCCL
            self._stream.wait_event(self._gate)
        with torch.cuda.stream(self._stream):
            b = self._collate(nxt)
            ev = torch.cuda.Event()
            ev.record(self._stream)
        b.__dict__["_ready"] = ev
        return b

    def current(self):
        b = self._next
        if self._stream is not None:
            self._gate = torch.cuda.Event()
            self._gate.record(torch.cuda.current_stream())
        ev = b.__dict__.pop("_ready", None) if (b is not None and self._stream is not None) else None
        if ev is not None:
            cur = torch.cuda.current_stream()
            cur.wait_event(ev)
            for t in _batch_tensors(b):          # allocated on the side stream, consumed on this one
                t.record_stream(cur)
        return b

    def advance(self):
        """Collate the following batch (call it right after the step's kernels have been enqueued)."""
        self._next = self._pull()

    def __iter__(self):
        while True:
            b = self.current()        # waits for the side stream's event: the batch is safe to use on the caller's stream
            if b is None:
                return
            yield b
            if self._next is b:       # the consumer did not call advance() itself
                self.advance()


def _batch_tensors(b):
    """Every device tensor a Batch1 owns (fields and K4 sort plans)."""
    def walk(v):
        if isinstance(v, torch.Tensor):
            if v.is_cuda:
                yield v
        elif isinstance(v, (tuple, list)):
            for x in v:
                yield from walk(x)
        elif isinstance(v, dict):
            for x in v.values():
                yield from walk(x)
    for k, v in b.__dict__.items():
        if k != "_dense":
            yield from walk(v)


class Batch1:
    """Same public surface as collator.py:149-215 (attributes, .to(device), len()); packed storage inside."""

    _REF_FIELDS = ("attn_bias", "attn_edge_type", "rel_pos", "spatial_pos", "in_degree", "out_degree", "x",
                   "edge_input", "adj", "adj1", "time", "time_normal", "cat", "poi_pos")

    def __init__(self, **kw):
        self.__dict__.update(kw)
        self.feature_matrix = None
        self._dense = {}

    def __len__(self):
        return int(self.B)

    @classmethod
    def from_dense(cls, ref, multi_hop_max_dist=20, rel_pos_max=1024, device=None):
        """A reference-collated dense batch (collator.py:149-215: padded int64 / fp32 tensors) -> the packed Batch1 the
        kernels consume.  Real nodes are the leading `x != 0` positions of every graph (pad_2d_squeeze, collator.py:29-37);
        everything is sliced to the real n_g x n_g block, so the padding the reference wrote is dropped, not copied.  Used
        when a caller hands `Graphormer.forward` the output of the reference's own collator."""
        from .algos import hop_stride
        dev = torch.device(device) if device is not None else ref.x.device
        t = lambda a: a.to(dev)
        x = t(ref.x)
        B, N = int(x.shape[0]), int(x.shape[1])
        nm = x.reshape(B, N, -1)[:, :, 0] != 0                                   # [B,N] real-node mask
        n = nm.sum(1).to(torch.int32)
        if bool(((torch.arange(N, device=dev).view(1, N) < n.view(B, 1)) != nm).any()):
            raise ValueError("Batch1.from_dense: real nodes must occupy the leading positions of every graph")
        pm = nm.unsqueeze(2) & nm.unsqueeze(1)                                   # [B,N,N] real-pair mask
        dk = int(multi_hop_max_dist)
        hops = hop_stride(dk)
        nl = n.long()
        zero = torch.zeros(1, dtype=torch.long, device=dev)
        sq_off = torch.cat([zero, torch.cumsum(nl * nl, 0)])
        node_off = torch.cat([zero, torch.cumsum(nl, 0)])
        tok_off = (node_off + torch.arange(B + 1, device=dev)).to(torch.int32)
        cells, Nn = int(sq_off[-1]), int(node_off[-1])
        rel = t(ref.rel_pos)[pm]
        ei = t(ref.edge_input)                                                   # [B,N,N,Dmax,1]
        Dm = min(int(ei.shape[3]), dk)
        edge_in8 = torch.zeros(cells, hops, dtype=torch.uint8, device=dev)
        edge_in8[:, :Dm] = ei[..., 0][pm][:, :Dm].to(torch.uint8)
        aet = t(ref.attn_edge_type)
        feat8 = aet.reshape(B, aet.shape[1], aet.shape[2], -1)[:, :N, :N, 0][pm].to(torch.uint8)
        g_of_node = torch.repeat_interleave(torch.arange(B, device=dev), nl)
        pos = torch.arange(Nn, device=dev) - node_off[:-1][g_of_node] + 1
        rows = torch.arange(Nn, device=dev) + g_of_node + 1
        Ntok = Nn + B
        tok_graph = torch.zeros(Ntok, dtype=torch.int32, device=dev)
        tok_pos = torch.zeros(Ntok, dtype=torch.int32, device=dev)
        tok_graph[rows] = g_of_node.int()
        tok_pos[rows] = pos.int()
        tok_graph[tok_off[:-1].long()] = torch.arange(B, device=dev, dtype=torch.int32)
        tn = t(ref.time_normal).reshape(B, N)[nm].float()
        maxdist = torch.zeros(B, dtype=torch.int32, device=dev)
        if cells:
            gcell = torch.repeat_interleave(torch.arange(B, device=dev), nl * nl)
            maxdist = torch.zeros(B, dtype=torch.long, device=dev).scatter_reduce(0, gcell, rel - 1, "amax").int()
        opt = lambda name: (t(getattr(ref, name)).reshape(B, N)[nm].int() if getattr(ref, name, None) is not None
                            else torch.zeros(Nn, dtype=torch.int32, device=dev))
        idx = getattr(ref, "idx", None)
        b = cls(B=B, N=int(n.max()) if B else 0, hops=hops, dk=dk, rel_pos_max=int(rel_pos_max), n_host=n.cpu().numpy(),
                h2d_bytes=0, n=n, sq_off=sq_off, node_off=node_off, tok_off=tok_off, tok_graph=tok_graph, tok_pos=tok_pos,
                feat8=feat8, x_nodes=x.reshape(B, N, -1)[:, :, 0][nm].int(), slot=(tn * 48).long().int(), time_nodes=opt("time"),
                time_normal_nodes=tn, cat_nodes=opt("cat"), in_deg=t(ref.in_degree)[nm].int(), out_deg=t(ref.out_degree)[nm].int(),
                user=t(ref.user).long().view(B, 1), y=t(ref.y).long().view(B),
                idx=t(torch.as_tensor(idx)).long() if idx is not None else torch.arange(B, device=dev),
                node_rows=rows, rel_pos16=rel.to(torch.int16), poi_pos16=t(ref.poi_pos)[pm].to(torch.int16), edge_in8=edge_in8,
                maxdist=maxdist, path16=None)
        return b

    def build_plans(self):
        """Fixed summation orders of the deterministic segmented scatter-adds (K4 backward): a stable sort of every key
        stream of the batch.  They depend on the batch indices only, so they are part of collation (device sorts, no
        host synchronisation); the category plan needs the model's cat_of_poi table and is added on first use."""
        from .ops import sort_plan
        plans = self.__dict__.setdefault("_plans", {})
        plans["node_rows"] = self.node_rows
        plans["poi"] = sort_plan(self.x_nodes.long() - 1)
        plans["slot"] = sort_plan(self.slot)
        plans["pos"] = sort_plan(self.tok_pos)
        ind = torch.zeros_like(self.tok_pos)
        ind[self.node_rows] = self.in_deg
        outd = torch.zeros_like(self.tok_pos)
        outd[self.node_rows] = self.out_deg
        plans["ind"] = sort_plan(ind)
        plans["outd"] = sort_plan(outd)
        # launch order of the attention kernels (mobgt_attn_fwd / _bwd `graph_order`): largest graph first
        self.size_order = torch.argsort(self.n, descending=True, stable=True).int()
        return plans

    def to(self, device):
        dev = torch.device(device)
        for k, v in list(self.__dict__.items()):
            if isinstance(v, torch.Tensor) and v.device != dev:
                self.__dict__[k] = v.to(dev, non_blocking=True)
        self._dense = {k: v.to(dev) for k, v in self._dense.items()}
        return self

    # ---- reference-shaped dense views (materialised lazily) ---------------------------------------
    def __getattr__(self, name):
        if name in Batch1._REF_FIELDS:
            d = self.__dict__.setdefault("_dense", {})
            if name not in d:
                d[name] = self._materialise(name)
            return d[name]
        raise AttributeError(name)

    def _sq_index(self):
        """(g, i, j) of every packed cell, as device int64 tensors."""
        if "_sqidx" not in self.__dict__:
            n = self.n.long()
            cells = n * n
            g = torch.repeat_interleave(torch.arange(self.B, device=n.device), cells)
            local = torch.arange(int(cells.sum()), device=n.device) - self.sq_off[:-1][g]
            self.__dict__["_sqidx"] = (g, local // n[g], local % n[g])
        return self.__dict__["_sqidx"]

    def _node_index(self):
        if "_nidx" not in self.__dict__:
            n = self.n.long()
            g = torch.repeat_interleave(torch.arange(self.B, device=n.device), n)
            q = torch.arange(int(n.sum()), device=n.device) - self.node_off[:-1][g]
            self.__dict__["_nidx"] = (g, q)
        return self.__dict__["_nidx"]

    def _materialise(self, name):
        B, N, dev = self.B, self.N, self.n.device
        if name in ("rel_pos", "spatial_pos", "poi_pos"):
            src = self.rel_pos16 if name != "poi_pos" else self.poi_pos16
            out = torch.zeros(B, N, N, dtype=torch.long, device=dev)
            g, i, j = self._sq_index()
            out[g, i, j] = src.long()
            return out
        if name == "edge_input":
            # hop axis = min(multi_hop_max_dist, max_g max(M_g))  (collator.py:323,366)
            dmax = int(min(getattr(self, "dk", self.hops), int(self.maxdist.max()))) if B else 0
            out = torch.zeros(B, N, N, dmax, 1, dtype=torch.long, device=dev)
            g, i, j = self._sq_index()
            out[g, i, j] = self.edge_in8[:, :dmax].long().unsqueeze(-1)
            return out
        if name == "attn_edge_type":
            out = torch.zeros(B, N + 1, N + 1, 1, dtype=torch.long, device=dev)
            g, i, j = self._sq_index()
            out[g, i, j, 0] = self.feat8.long()
            return out
        if name in ("adj", "adj1"):
            T = N + 1 if name == "adj" else N
            out = torch.zeros(B, T, T, dtype=torch.bool, device=dev)
            g, i, j = self._sq_index()
            out[g, i, j] = self.feat8 != 0
            if name == "adj":          # wrapper.py:79-81: the virtual token row/col sits at index n_g
                ar = torch.arange(B, device=dev)
                n = self.n.long()
                for gi in range(B):
                    out[gi, n[gi], :n[gi] + 1] = True
                    out[gi, :n[gi] + 1, n[gi]] = True
                del ar
            return out
        if name == "attn_bias":
            T = N + 1
            out = torch.zeros(B, T, T, dtype=torch.float, device=dev)
            col = torch.arange(T, device=dev).view(1, 1, T)
            out.masked_fill_(col > self.n.long().view(B, 1, 1), float("-inf"))            # collator.py:57-64
            if self.rel_pos_max <= 510:
                g, i, j = self._sq_index()
                m = (self.rel_pos16.long() - 1) >= self.rel_pos_max                      # collator.py:354-358
                out[g[m], i[m] + 1, j[m] + 1] = float("-inf")
            return out
        g, q = self._node_index()
        if name in ("in_degree", "out_degree"):
            out = torch.zeros(B, N, dtype=torch.long, device=dev)
            out[g, q] = (self.in_deg if name == "in_degree" else self.out_deg).long()
            return out
        if name in ("x", "time", "cat"):
            src = {"x": self.x_nodes, "time": self.time_nodes, "cat": self.cat_nodes}[name]
            out = torch.zeros(B, N, 1, dtype=torch.long, device=dev)
            out[g, q, 0] = src.long()
            return out
        if name == "time_normal":
            out = torch.zeros(B, N, 1, dtype=torch.float, device=dev)
            out[g, q, 0] = self.time_normal_nodes
            return out
        raise AttributeError(name)


class HostPack:
    """The host half of a collated batch: every host-packed array laid out in ONE byte buffer (16-byte aligned segments),
    plus the few Python scalars the device half needs.  Pure numpy: safe to build in DataLoader worker processes, cheap to
    ship through shared memory, and uploaded with a single H2D copy."""

    def __init__(self, buf, layout, B, N, ns, cells, padded=False):
        self.buf, self.layout, self.B, self.N, self.ns, self.cells, self.padded = buf, layout, B, N, ns, cells, padded


def _bucket_sizes(ntok, cells, nmax, B, large_graphs=False):
    """Bucketed (tokens, cells, max nodes): tokens to a multiple of 512 (GEMM rows: the cost that scales), cells to a power
    of two (memory only), the node cap to a power of two (tile counts of K2 / K3), at most 512 — or 1024 with large_graphs."""
    ntok_b = max(512, (ntok + 511) // 512 * 512)
    cells_b = 4096
    while cells_b < cells:
        cells_b *= 2
    n_b = 8
    while n_b < nmax:
        n_b *= 2
    return ntok_b, cells_b, min(n_b, _node_cap(large_graphs))


def _host_plan(keys):
    """Stable sort of an int key stream -> (perm i32, sorted keys i32): ops.sort_plan on the host."""
    k = np.ascontiguousarray(keys)
    small = k.size == 0 or (int(k.min()) >= 0 and int(k.max()) < 65536)
    perm = np.argsort(k.astype(np.uint16) if small else k.astype(np.int64), kind="stable").astype(np.int32)   # 16-bit keys: radix sort
    return perm, k[perm].astype(np.int32)


def _node_cap(large_graphs):
    return _C.MAX_MODEL_NODES if large_graphs else _C.MAX_NODES


def _check_node_cap(ns, large_graphs):
    """The model's kernels (K2 / K3) take graphs of up to MAX_NODES = 512 nodes, and of up to MAX_MODEL_NODES = 1024 in the
    opt-in large_graphs mode (K1 alone takes 1024 either way)."""
    cap = _node_cap(large_graphs)
    if len(ns) and int(np.max(ns)) > cap:
        hint = "" if large_graphs else f" (large_graphs=True takes up to {_C.MAX_MODEL_NODES})"
        raise ValueError(f"node counts must be in [1, {cap}]{hint}")


def pack_host(items, max_node=512, bucket=False, large_graphs=False):
    """raw dataset items (owndata.py:340-349 fields; numpy or torch) -> HostPack.  No CUDA, no torch ops on the hot path.

    bucket=True pads the per-token / per-node / per-cell arrays to bucket sizes (`_bucket_sizes`): padding tokens are extra
    "graph tokens" that belong to no graph (no tok_off range covers them, so attention never reads or writes them and their
    gradient is exactly zero), padding nodes map to them one to one with padding-row indices, padding cells are never indexed.
    Per-graph sizes (n, offsets) are untouched, so every result for the real graphs is identical to the unpadded batch.
    large_graphs: see `collate_from_host` (here it only lets the bucketed node cap reach 1024)."""
    items = [it for it in items if it is not None and len(_to_np(it.x)) <= max_node]     # collator.py:313
    B = len(items)
    ns = np.array([len(_to_np(it.x)) for it in items], np.int32)
    sq = np.zeros(B + 1, np.int64)
    np.cumsum(ns.astype(np.int64) ** 2, out=sq[1:])
    no = np.zeros(B + 1, np.int64)
    np.cumsum(ns.astype(np.int64), out=no[1:])
    Nn, cells = int(no[-1]), int(sq[-1])
    # all edge lists of the batch in one shot (one scatter / two bincounts instead of a Python loop over the items)
    eis = [_to_np(it.edge_index) for it in items]
    ecnt = np.array([e.shape[1] for e in eis], np.int64)
    ei = np.concatenate(eis, axis=1).astype(np.int64) if B else np.zeros((2, 0), np.int64)
    ea = np.concatenate([_to_np(it.edge_attr).reshape(-1) for it in items]).astype(np.int64) if B else np.zeros(0, np.int64)
    eg = np.repeat(np.arange(B), ecnt)                    # graph of every edge
    indeg = np.bincount(no[:-1][eg] + ei[0], minlength=Nn).astype(np.int32)   # wrapper.py:97: adj.sum(dim=1)
    outdeg = np.bincount(no[:-1][eg] + ei[1], minlength=Nn).astype(np.int32)  # wrapper.py:98: adj.sum(dim=0)
    # the reference indexes nn.Embedding(128, ...) tables with these (edge_encoder :784, in/out_degree_encoder :861-862) and
    # raises IndexError past row 127; fail the same way here instead of wrapping in uint8 / reading out of bounds on the device
    if len(ea) and (ea.min() < 0 or ea.max() + 3 >= 128):
        raise IndexError(f"edge_attr {int(ea.max())}: edge_input index edge_attr+3 must stay below the 128 rows of edge_encoder")
    if Nn and max(int(indeg.max()), int(outdeg.max())) + 1 >= 128:
        raise IndexError(f"node degree {max(int(indeg.max()), int(outdeg.max()))}: degree+1 must stay below the 128 rows of "
                         "in_degree_encoder / out_degree_encoder")

    def cat_field(name, dtype):
        return np.concatenate([_to_np(getattr(it, name)).reshape(-1) for it in items]).astype(dtype, copy=False)

    x_nodes = cat_field("x", np.int32)
    tn = cat_field("time_normal", np.float32)
    time_nodes = cat_field("time", np.int32)
    cat_nodes = cat_field("cat", np.int32)
    slot = (tn * np.float32(48)).astype(np.int64).astype(np.int32)          # model_fqandtoyo.py:1262
    user = (np.array([_to_np(it.user).reshape(-1)[0] for it in items]).astype(np.int64) + 1).reshape(B, 1)   # wrapper.py:39
    y = np.array([_to_np(it.y).reshape(-1)[0] for it in items]).astype(np.int64)                             # collator.py:367
    idx = np.array([int(getattr(it, "idx", i)) for i, it in enumerate(items)], np.int64)
    tok_off = (no + np.arange(B + 1)).astype(np.int32)
    g_of_node = np.repeat(np.arange(B, dtype=np.int32), ns)
    pos_of_node = (np.arange(Nn) - no[:-1][g_of_node] + 1).astype(np.int32)
    Ntok = Nn + B
    tok_graph = np.zeros(Ntok, np.int32)
    tok_pos = np.zeros(Ntok, np.int32)
    rows = np.arange(Nn) + g_of_node + 1
    tok_graph[rows] = g_of_node
    tok_pos[rows] = pos_of_node
    tok_graph[tok_off[:-1]] = np.arange(B)
    in_deg, out_deg, node_rows = indeg + 1, outdeg + 1, rows.astype(np.int64)    # pad_1d_unsqueeze "+1" (collator.py:12)
    N_out, cells_alloc, padded = (int(ns.max()) if B else 0), cells, False
    if bucket and B:
        ntok_b, cells_alloc, N_out = _bucket_sizes(Ntok, cells, int(ns.max()), B, large_graphs)
        pad = ntok_b - Ntok                                   # padding tokens == padding nodes (Ntok = Nn + B)
        if pad or cells_alloc != cells or N_out != int(ns.max()):
            padded = True
            z32 = np.zeros(pad, np.int32)
            tok_graph, tok_pos = np.concatenate([tok_graph, z32]), np.concatenate([tok_pos, z32])
            x_nodes = np.concatenate([x_nodes, np.ones(pad, np.int32)])
            slot, time_nodes = np.concatenate([slot, z32]), np.concatenate([time_nodes, z32])
            tn = np.concatenate([tn, np.zeros(pad, np.float32)])
            cat_nodes = np.concatenate([cat_nodes, np.ones(pad, np.int32)])
            in_deg, out_deg = np.concatenate([in_deg, z32]), np.concatenate([out_deg, z32])      # 0 = the padding row
            node_rows = np.concatenate([node_rows, Ntok + np.arange(pad, dtype=np.int64)])
    host = dict(n=ns, sq_off=sq, node_off=no, tok_off=tok_off, tok_graph=tok_graph, tok_pos=tok_pos, feat8=None,
                x_nodes=x_nodes, slot=slot, time_nodes=time_nodes, time_normal_nodes=tn, cat_nodes=cat_nodes,
                in_deg=in_deg, out_deg=out_deg, user=user, y=y, idx=idx, node_rows=node_rows)
    # The fixed summation orders of the K4 backward (stable sorts of the batch's key streams, Batch1.build_plans) and the launch
    # order of the attention kernels depend on the indices only: they are built HERE, in the loader's worker process (numpy radix
    # sorts of 16-bit keys, ~1 ms per batch off the critical path), and ride along in the one H2D copy — instead of ~25 device
    # sort / scatter kernels per batch running next to the training step.
    ind_tok = np.zeros(len(tok_pos), np.int32)
    ind_tok[node_rows] = in_deg
    outd_tok = np.zeros(len(tok_pos), np.int32)
    outd_tok[node_rows] = out_deg
    for name, keys in (("poi", x_nodes - 1), ("slot", slot), ("pos", tok_pos), ("ind", ind_tok), ("outd", outd_tok)):
        perm, ks = _host_plan(keys)
        host[f"plan_{name}_perm"], host[f"plan_{name}_keys"] = perm, ks
    host["size_order"] = np.argsort(-ns.astype(np.int64), kind="stable").astype(np.int32)
    layout, total = {}, 0
    for k, a in host.items():
        if k == "feat8":
            shape, dt, nbytes = (cells_alloc,), np.dtype(np.uint8), cells_alloc
        else:
            a = np.ascontiguousarray(a)
            host[k] = a
            shape, dt, nbytes = a.shape, a.dtype, a.nbytes
        layout[k] = (total, shape, dt.str, nbytes)
        total += (nbytes + 15) // 16 * 16
    buf = np.zeros(max(total, 16), np.uint8)
    for k, a in host.items():
        if a is not None:
            off, _, _, nbytes = layout[k]
            buf[off:off + nbytes] = a.reshape(-1).view(np.uint8)
    # the edge-type plane is scattered straight into its segment of the buffer
    off = layout["feat8"][0]
    buf[off + sq[:-1][eg] + ei[0] * ns.astype(np.int64)[eg] + ei[1]] = ea + 2     # wrapper.py:49-53: convert_to_single_emb(+1) then +1
    return HostPack(buf, layout, B, N_out, ns, cells_alloc, padded)


def _upload_pack(hp, dev):
    """HostPack -> name -> device tensor views (one async H2D copy from pinned memory)."""
    total = int(hp.buf.shape[0])
    src = hp.buf.numpy() if isinstance(hp.buf, torch.Tensor) else hp.buf      # worker batches arrive as shared-memory tensors
    st = _staging.setdefault(str(dev), _Staging())
    slot, pinned = st.get(total)
    pinned.numpy()[:total] = src              # plain memcpy into the persistent pinned staging buffer (numpy: no thread-pool launch)
    dbuf = torch.empty(total, dtype=torch.uint8, device=dev)
    dbuf.copy_(pinned[:total], non_blocking=True)
    st.mark(slot)
    out = {}
    for k, (off, shape, dts, nbytes) in hp.layout.items():
        tdt = torch.from_numpy(np.zeros(0, np.dtype(dts))).dtype
        out[k] = dbuf[off:off + nbytes].view(tdt).view(tuple(shape))
    return out


def collate_from_host(hp, world=None, latlon_dev=None, multi_hop_max_dist=20, rel_pos_max=1024, device="cuda", want_path=False,
                      large_graphs=False):
    """The device half of collation: one H2D copy, the K4-backward sort plans, K1 (APSP + path edges) and poi_pos.
    Graphs above 512 nodes raise ValueError unless large_graphs=True, which takes up to 1024 (T <= 1025 tokens: the
    attention-bias and attention kernels run such graphs on their large-graph paths)."""
    _check_node_cap(hp.ns.numpy() if isinstance(hp.ns, torch.Tensor) else hp.ns, large_graphs)
    _C.require_cuda()
    dev = torch.device(device)
    views = _upload_pack(hp, dev)
    ns = hp.ns.numpy() if isinstance(hp.ns, torch.Tensor) else hp.ns
    dk = int(multi_hop_max_dist)
    hops = hop_stride(dk)                  # bytes per edge_in8 row; slots [dk, hops) are padding
    h2d_bytes = int(sum(v.numel() * v.element_size() for v in views.values()))
    plans = {k[5:]: views.pop(k) for k in list(views) if k.startswith("plan_")}          # built by pack_host on the host
    size_order = views.pop("size_order", None)
    b = Batch1(B=hp.B, N=hp.N, hops=hops, dk=dk, rel_pos_max=int(rel_pos_max), n_host=ns, h2d_bytes=h2d_bytes, padded=bool(hp.padded), **views)
    if plans:
        b.__dict__["_plans"] = {name: (plans[f"{name}_perm"], plans[f"{name}_keys"]) for name in ("poi", "slot", "pos", "ind", "outd")}
        b.__dict__["_plans"]["node_rows"] = b.node_rows
        b.size_order = size_order
    else:
        b.build_plans()
    k1 = apsp_edge_input_packed(b.feat8, b.n, b.sq_off, ns, hops=hops, shift=1, want_path=want_path, dk=dk)
    b.rel_pos16, b.edge_in8, b.maxdist, b.path16 = k1["dist"], k1["edge_in"], k1["maxdist"], k1["path"]
    b.poi_pos16 = torch.empty(hp.cells, dtype=torch.int16, device=dev)
    if world is not None:
        if latlon_dev is None:
            latlon_dev = torch.from_numpy(world.latlon).to(dev)
        b._latlon = latlon_dev
        _C.call("mobgt_poi_pos", _C.ptr(b.x_nodes), _C.ptr(b.n), _C.ptr(b.sq_off), _C.ptr(b.node_off), _C.ptr(latlon_dev),
                float(np.float32(world.dist_max)), int(world.num_bins), hp.B, int(b.N), _C.ptr(b.poi_pos16), _C.stream_ptr())
    else:
        b.poi_pos16.fill_(1)
    return b


def collate_packed(items, world=None, latlon_dev=None, max_node=512, multi_hop_max_dist=20, rel_pos_max=1024,
                   device="cuda", want_path=False, bucket=False, large_graphs=False):
    """Shared body of the three POI collators.  items: raw dataset items (owndata.py:340-349 fields; numpy or
    torch).  Returns a device-resident Batch1.  bucket: see `pack_host` (training loaders; the reference-shaped dense views
    of a bucketed batch are padded to the bucket's node cap instead of the batch maximum)."""
    _C.require_cuda()
    return collate_from_host(pack_host(items, max_node, bucket=bucket, large_graphs=large_graphs), world, latlon_dev,
                             multi_hop_max_dist, rel_pos_max, device, want_path, large_graphs)


def collator_foursquare(items, max_node=512, multi_hop_max_dist=20, rel_pos_max=20, world=None, latlon_dev=None, **kw):
    """collator.py:310-458"""
    return collate_packed(items, world, latlon_dev, max_node, multi_hop_max_dist, rel_pos_max, **kw)


def collator_gowalla(items, max_node=512, multi_hop_max_dist=20, rel_pos_max=20, world=None, latlon_dev=None, **kw):
    """collator.py:460-608"""
    return collate_packed(items, world, latlon_dev, max_node, multi_hop_max_dist, rel_pos_max, **kw)


def collator_toyota(items, max_node=512, multi_hop_max_dist=20, rel_pos_max=20, world=None, latlon_dev=None, **kw):
    """collator.py:610-748"""
    return collate_packed(items, world, latlon_dev, max_node, multi_hop_max_dist, rel_pos_max, **kw)
