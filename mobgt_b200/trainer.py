"""The training / evaluation loop of the MobGT hot path — what `pytorch_lightning.Trainer` + DDP do for the reference
(entry.py:141-161): data parallel over trajectory graphs, one process per GPU.

    tr = Trainer(model, device, world_size)            # flat fp32 gradient buffer, AdamW + PolynomialDecayLR, CUDA graphs
    loss = tr.train_step(batch)                        # zero grads, forward, loss, backward, all-reduce, optimizer, schedule
    metrics = tr.evaluate(batches)                     # fused K5 head per batch, metric sums all-reduced once

Both `mobgt_b200.entry` (the reference's command line) and `bench.py` drive THIS class, so the benchmarked step is the one the
public entry point runs.

* Gradients live in ONE flat fp32 buffer (`parallel.FlatGrads`): the data-parallel exchange is a single NCCL all-reduce, and
  `1 / world` is folded into it (ReduceOp.AVG).
* Forward + backward of a batch shape that repeats is captured in a CUDA graph (`graphs.GraphedTrainStep`) and replayed;
  a shape is captured when it is seen for the second time, other shapes run eagerly (same kernels, ~550 launches).
* With world_size > 1 and `overlap=True` an EAGER step all-reduces the gradient of `out_proj.weight` — 77 of the 92 MB at
  P = 60 000 and the FIRST gradient the backward produces — on a side stream as soon as it is complete, while the encoder
  backward is still running; the remainder of the buffer follows at the end of the backward.  A graph-replayed step issues one
  flat all-reduce after the replay: capturing the NCCL collective inside the graph (`overlap_in_graph=True`) was measured on
  2 x B200 (profiles/r2/r2g_bench_n2_*.json): 6.68 ms/step against 6.65 ms without it, and the process then hung in
  destroy_process_group — so it is off by default.
"""
import os
import sys

import torch
import torch.distributed as dist

from . import _C, graphs, ops, parallel


def _signature(batch):
    return (int(batch.B), int(batch.N), int(batch.tok_pos.numel()), int(batch.rel_pos16.numel()), int(batch.hops),
            int(getattr(batch, "dk", batch.hops)), bool(getattr(batch, "padded", False)), ops.all_large(batch))


class Trainer:
    def __init__(self, model, device, world_size=1, cuda_graph=True, overlap=True, overlap_in_graph=False, max_graphs=16, group=None):
        self.model, self.dev, self.world, self.group = model, torch.device(device), int(world_size), group
        (self.opt,), (cfg,) = model.configure_optimizers()
        self.sched = cfg["scheduler"]
        if hasattr(self.opt, "flat_grad"):      # optim.FlatAdamW owns the flat buffers (p.data / p.grad are views of them)
            self.flat = self.opt.flat_grad
        else:
            self.grads = parallel.FlatGrads(model.parameters(), self.dev)
            self.flat = self.grads.flat
        self.use_graph, self.max_graphs = bool(cuda_graph), int(max_graphs)
        self._graphs, self._seen, self._no_capture = {}, {}, set()
        self._pool = torch.cuda.graph_pool_handle() if cuda_graph else None      # one memory pool for all captured shapes
        self.eager_steps = self.graph_steps = 0
        self.step_count = 0
        self.graph_note = "off" if not cuda_graph else "eager (no shape repeated yet)"
        # ---- overlapped all-reduce: bucket 0 = the gradient slice of out_proj.weight, bucket 1 = everything else
        self._overlap = bool(overlap) and self.world > 1
        self._side = torch.cuda.Stream(device=self.dev) if self._overlap else None
        self._early = None
        self._early_done, self._early_joined, self._overlap_in_graph = None, False, bool(overlap_in_graph)
        self._constructing = False
        # data parallel + CUDA graphs: the step is captured as two graphs cut behind the head backward, and the all-reduce of
        # the out_proj bucket runs on the side stream under the second one (MOBGT_SPLIT_GRAPH=0: one graph, one flat all-reduce)
        self._split_graph = self._overlap and hasattr(model, "out_proj") and os.environ.get("MOBGT_SPLIT_GRAPH", "1") != "0"
        if self._overlap and hasattr(model, "out_proj"):
            w = model.out_proj.weight
            off = (w.grad.data_ptr() - self.flat.data_ptr()) // 4
            self._early = (int(off), int(off) + w.numel())
            ops.on_grad_ready(w, self._on_head_grad)          # fired by the head Linear's backward (ops.LinearBiasFn)

    # ---------------------------------------------------------------------------------------- gradient exchange
    def _on_head_grad(self, _param):
        """out_proj.weight.grad is final (its only use is the head GEMM): start its all-reduce now, on the side stream.
        Under CUDA-graph capture the side stream joins the capture, so the collective becomes a node of the graph."""
        capturing = torch.cuda.is_current_stream_capturing()
        if not self._overlap or (capturing and not self._overlap_in_graph) or (self._constructing and not capturing):
            return          # (the eager warm-up passes of a graph capture issue no collective: capture stays rank-local)
        ev = torch.cuda.Event()
        ev.record(torch.cuda.current_stream())
        self._side.wait_event(ev)
        a, b = self._early
        with torch.cuda.stream(self._side):
            dist.all_reduce(self.flat[a:b], op=dist.ReduceOp.AVG, group=self.group)
            done = torch.cuda.Event()
            done.record(self._side)
        self._early_done = done

    def _start_early_allreduce(self):
        """All-reduce the out_proj bucket on the side stream, ordered after everything enqueued on the training stream."""
        ev = torch.cuda.Event()
        ev.record(torch.cuda.current_stream())
        self._side.wait_event(ev)
        a, b = self._early
        with torch.cuda.stream(self._side):
            dist.all_reduce(self.flat[a:b], op=dist.ReduceOp.AVG, group=self.group)
            done = torch.cuda.Event()
            done.record(self._side)
        self._early_done = done

    def _join_early(self):
        """Right after backward (also inside a graph capture): the training stream waits for the early all-reduce."""
        if self._early_done is not None:
            torch.cuda.current_stream().wait_event(self._early_done)
            self._early_done = None
            self._early_joined = True

    def _exchange(self, early_done):
        """All-reduce (mean) whatever part of the flat gradient buffer the early bucket has not covered."""
        if self.world <= 1:
            return
        if self._early is None or not early_done:
            dist.all_reduce(self.flat, op=dist.ReduceOp.AVG, group=self.group)
            return
        a, b = self._early
        if a > 0:
            dist.all_reduce(self.flat[:a], op=dist.ReduceOp.AVG, group=self.group)
        if b < self.flat.numel():
            dist.all_reduce(self.flat[b:], op=dist.ReduceOp.AVG, group=self.group)

    # ---------------------------------------------------------------------------------------- one step
    def _graph_for(self, batch):
        # a batch holding a graph of more than 512 nodes (collator large_graphs mode, at most one such graph in a few thousand)
        # runs eagerly: its bias and dS planes are ~40x those of an ordinary batch and would stay reserved in the graph pool
        if not self.use_graph or int(batch.N) > _C.MAX_NODES:
            return None
        sig = _signature(batch)
        g = self._graphs.get(sig)
        if g is not None or sig in self._no_capture:
            return g
        self._seen[sig] = self._seen.get(sig, 0) + 1
        if self._seen[sig] < 2 or len(self._graphs) >= self.max_graphs:
            return None
        g = None
        for in_graph in ((True, False) if (self._overlap and self._overlap_in_graph) else (self._overlap_in_graph,)):
            self._overlap_in_graph = in_graph
            self._early_done, self._early_joined = None, False
            self._constructing = True
            try:
                g = graphs.GraphedTrainStep(self.model, self.flat, batch, after_backward=self._join_early, pool=self._pool,
                                            split_head=self._split_graph)
                g.early_in_graph = bool(self._early_joined)
                self._graphs[sig] = g
                self.graph_note = "fwd+bwd captured" + (" (+ early all-reduce of out_proj.weight.grad in-graph)" if g.early_in_graph else "") \
                    + (" as two graphs cut behind the head backward; the out_proj bucket is all-reduced under the second" if g.split else "")
                break
            except graphs.GraphCaptureError as e:
                if os.environ.get("MOBGT_STRICT_GRAPH") == "1":
                    raise
                self.graph_note = f"eager ({str(e)[:400]})"
                print(f"[mobgt] CUDA-graph capture failed, running eagerly: {e}", file=sys.stderr)
                g = None
            finally:
                self._constructing = False
        if g is None:
            self._no_capture.add(sig)
        return g

    def forward_backward(self, batch):
        """zero grads + forward + loss + backward (graph replay when the shape has been captured).  -> loss tensor"""
        g = self._graph_for(batch)
        if g is not None:
            try:
                g.load(batch)
                if g.split and self._early is not None:
                    loss = g.run_a()
                    self._start_early_allreduce()          # out_proj.weight.grad is final: its bucket leaves now ...
                    g.run_b()                              # ... while the encoder backward runs
                    self._join_early()
                    self.graph_steps += 1
                    return loss.detach(), True
                loss = g.run()
                self.graph_steps += 1
                return loss.detach(), g.early_in_graph
            except graphs.ShapeMismatch:
                pass
        self.eager_steps += 1
        self.flat.zero_()
        ops.grads_zeroed(self.flat)
        self._early_done, self._early_joined = None, False
        loss = self.model.training_step(batch)
        loss.backward()
        self._join_early()
        # detached: a live reference to the autograd graph would keep this step's AccumulateGrad nodes (bound to the stream
        # they were created on) alive into the next step — fatal for a later CUDA-graph capture on another stream
        return loss.detach(), self._early_joined

    def train_step(self, batch):
        loss, early_done = self.forward_backward(batch)
        self._exchange(early_done)
        self.opt.step()
        self.sched.step()
        self.step_count += 1
        return loss

    @property
    def graph_launches(self):
        """libmobgt kernel nodes per replay of the (first) captured graph."""
        for g in self._graphs.values():
            return g.launches
        return 0

    # ---------------------------------------------------------------------------------------- evaluation
    def evaluate(self, batches, vocab_parallel=False, quiet=False):
        """model_fqandtoyo.py:1530-1597 over an iterable of batches (this rank's shard): every batch goes through the fused
        K5 head; the metric SUMS of all ranks are all-reduced once."""
        was_training = self.model.training
        self.model.eval()
        outs = []
        with torch.no_grad():
            for b in batches:
                outs.append(self.model.test_step(b, vocab_parallel=(self.group or dist.group.WORLD) if
                                                 (vocab_parallel and self.world > 1) else None))
        res = self.model.test_epoch_end(outs, group=self.group, quiet=quiet)
        self.model.train(was_training)
        return res

    # ---------------------------------------------------------------------------------------- checkpoints (entry.py:123-137)
    def state_dict(self):
        return {"state_dict": self.model.state_dict(), "optimizer": self.opt.state_dict(), "lr_scheduler": self.sched.state_dict(),
                "global_step": self.step_count}

    def load_state_dict(self, ck, with_optimizer=True):
        self.model.load_state_dict(ck["state_dict"], strict=False)
        if with_optimizer and "optimizer" in ck:
            self.opt.load_state_dict(ck["optimizer"])
            self.sched.load_state_dict(ck["lr_scheduler"])
            self.step_count = int(ck.get("global_step", 0))
