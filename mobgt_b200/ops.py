"""torch-facing wrappers of the libmobgt kernels: raw calls + autograd.Function pairs.

PyTorch is plumbing here (device memory, streams, autograd graph); the arithmetic of the hot ops is in
mobgt_b200/csrc/*.cu behind the C-ABI (include/mobgt.h).  No op has a torch/CPU fallback.
"""
import torch

from . import _C

F32, BF16 = 0, 1
NUM_HEADS = 8            # the canonical shape's head count
BIAS_HEADS = (8, 12)     # head counts the attention-bias kernels are built for (csrc/k2_bias.cu K2Heads)
HEAD_DIM = 24            # the canonical shape's head dim (hidden 128: (128 + 64) / 8)
HEAD_DIMS = (16, 24)     # head dims the attention kernels are built for (csrc/k3_small.cuh AttnShape)


def _dt(t):
    if t.dtype == torch.float32:
        return F32
    if t.dtype == torch.bfloat16:
        return BF16
    raise _C.MobgtError(f"unsupported dtype {t.dtype}")


def bias_pitch(T):
    """Row pitch (elements) of the bias planes: a multiple of 8 so that rows are 16-byte aligned for TMA."""
    return (T + 7) // 8 * 8


# ----------------------------------------------------------------------------------------------- K2
def _dk(batch):
    """multi_hop_max_dist of a batch (hop slots that are live); batch.hops is the byte stride of its edge_in8 rows."""
    return int(getattr(batch, "dk", batch.hops))


def bias_fwd_raw(batch, R, Ppos, E, W, tvd, out_dtype=torch.bfloat16, T=None, Tp=None):
    B, H = batch.B, R.shape[1]
    T = T or batch.N + 1
    Tp = Tp or bias_pitch(T)
    dev = R.device
    out = torch.empty(B, H, T, Tp, dtype=out_dtype, device=dev)
    ws_bytes = int(_C.lib().mobgt_bias_fwd_workspace_bytes(batch.hops, H))
    if ws_bytes < 0:
        raise _C.MobgtError(f"mobgt_bias_fwd_workspace_bytes rejected hops={batch.hops} H={H}")
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    _C.call("mobgt_bias_fwd", _C.ptr(batch.n), _C.ptr(batch.sq_off), _C.ptr(batch.rel_pos16), _C.ptr(batch.poi_pos16),
            _C.ptr(batch.edge_in8), B, T, Tp, batch.hops, _dk(batch), H, batch.rel_pos_max, int(Ppos.shape[0]), _C.ptr(R), _C.ptr(Ppos),
            _C.ptr(E), _C.ptr(W), _C.ptr(tvd), _C.ptr(ws), _C.ptr(out), _dt(out), _C.stream_ptr())
    return out


def bias_bwd_raw(batch, dbias, E, W, num_bins):
    """dbias: f32 [B,H,T,Tp] (sum over layers) or bf16 [L,B,H,T,Tp] (per-layer dS planes, summed in the kernel)."""
    if dbias.dtype == torch.bfloat16:
        L, B, H, T, Tp = dbias.shape
        dt, stride = BF16, dbias.stride(0)
    else:
        B, H, T, Tp = dbias.shape
        L, dt, stride = 1, F32, 0
    dev = dbias.device
    hops = batch.hops
    ws_bytes = int(_C.lib().mobgt_bias_bwd_heads_workspace_bytes(T, hops, num_bins, H))
    if ws_bytes < 0:
        raise _C.MobgtError(f"mobgt_bias_bwd_heads_workspace_bytes rejected T={T} hops={hops} num_bins={num_bins} H={H}")
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    dR = torch.empty(512, H, dtype=torch.float32, device=dev)
    dP = torch.empty(num_bins, H, dtype=torch.float32, device=dev)
    dE = torch.empty(128, H, dtype=torch.float32, device=dev)
    dW = torch.zeros(W.numel(), dtype=torch.float32, device=dev)   # rows >= hops*H*H of edge_dis_encoder get no gradient
    dtv = torch.empty(H, dtype=torch.float32, device=dev)
    _C.call("mobgt_bias_bwd", _C.ptr(batch.n), _C.ptr(batch.sq_off), _C.ptr(batch.rel_pos16), _C.ptr(batch.poi_pos16),
            _C.ptr(batch.edge_in8), B, T, Tp, hops, _dk(batch), H, batch.rel_pos_max, num_bins, _C.ptr(dbias), dt, L, stride, _C.ptr(E),
            _C.ptr(W), _C.ptr(ws), ws_bytes, _C.ptr(dR), _C.ptr(dP), _C.ptr(dE), _C.ptr(dW), _C.ptr(dtv), _C.stream_ptr())
    return dR, dP, dE, dW.view_as(W), dtv


def bias_direct_fwd_raw(batch, R, Ppos, E, tvd, out_dtype=torch.bfloat16, T=None, Tp=None):
    """K2 for the direct edge encoding (edge_type other than multi_hop): the edge term of a pair is E[attn_edge_type], read from
    the batch's feat8 plane.  Same output layout as bias_fwd_raw."""
    B, H = batch.B, R.shape[1]
    T = T or batch.N + 1
    Tp = Tp or bias_pitch(T)
    out = torch.empty(B, H, T, Tp, dtype=out_dtype, device=R.device)
    _C.call("mobgt_bias_direct_fwd", _C.ptr(batch.n), _C.ptr(batch.sq_off), _C.ptr(batch.rel_pos16), _C.ptr(batch.poi_pos16),
            _C.ptr(batch.feat8), B, T, Tp, H, batch.rel_pos_max, int(Ppos.shape[0]), _C.ptr(R), _C.ptr(Ppos), _C.ptr(E), _C.ptr(tvd),
            _C.ptr(out), _dt(out), _C.stream_ptr())
    return out


def bias_direct_bwd_raw(batch, dbias, num_bins):
    """Backward of bias_direct_fwd_raw from the same dbias forms as bias_bwd_raw -> (dR, dPpos, dE, dtvd); dE row 0 is 0."""
    if dbias.dtype == torch.bfloat16:
        L, B, H, T, Tp = dbias.shape
        dt, stride = BF16, dbias.stride(0)
    else:
        B, H, T, Tp = dbias.shape
        L, dt, stride = 1, F32, 0
    dev = dbias.device
    ws_bytes = int(_C.lib().mobgt_bias_direct_bwd_workspace_bytes(T, num_bins, H))
    if ws_bytes < 0:
        raise _C.MobgtError(f"mobgt_bias_direct_bwd_workspace_bytes rejected T={T} num_bins={num_bins} H={H}")
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    dR = torch.empty(512, H, dtype=torch.float32, device=dev)
    dP = torch.empty(num_bins, H, dtype=torch.float32, device=dev)
    dE = torch.empty(128, H, dtype=torch.float32, device=dev)
    dtv = torch.empty(H, dtype=torch.float32, device=dev)
    _C.call("mobgt_bias_direct_bwd", _C.ptr(batch.n), _C.ptr(batch.sq_off), _C.ptr(batch.rel_pos16), _C.ptr(batch.poi_pos16),
            _C.ptr(batch.feat8), B, T, Tp, H, batch.rel_pos_max, num_bins, _C.ptr(dbias), dt, L, stride, _C.ptr(ws), ws_bytes,
            _C.ptr(dR), _C.ptr(dP), _C.ptr(dE), _C.ptr(dtv), _C.stream_ptr())
    return dR, dP, dE, dtv


def _bias_fwd(batch, direct, R, Ppos, E, W, tvd, out_dtype):
    """K2 forward of either edge encoding; the tables are fp32 contiguous (W is not read by the direct encoding)."""
    if direct:
        return bias_direct_fwd_raw(batch, R, Ppos, E, tvd.view(-1), out_dtype)
    return bias_fwd_raw(batch, R, Ppos, E, W.view(-1), tvd.view(-1), out_dtype)


def _bias_bwd(batch, direct, dbias, E, W, num_bins):
    """-> the gradients of (R, Ppos, E, W, tvd) as the autograd nodes return them; W's is None for the direct encoding."""
    if direct:
        dR, dP, dE, dt = bias_direct_bwd_raw(batch, dbias, num_bins)
        dW = None
    else:
        dR, dP, dE, dW, dt = bias_bwd_raw(batch, dbias, E, W.view(-1), num_bins)
        dW = dW.view(-1, 1)
    dR[0].zero_()          # padding_idx rows (never indexed by a packed pair anyway)
    dP[0].zero_()
    return dR, dP, dE, dW, dt.view(1, -1)


class AttnBias(torch.autograd.Function):
    """graph_attn_bias = f(rel_pos, poi_pos, edge_input; 5 tables)   (model_fqandtoyo.py:1143-1216) as a stand-alone
    differentiable op (gradient: a plain [B,H,T,Tp] tensor).  The model's forward uses BiasLink below, whose backward
    consumes the per-layer bf16 dS planes of the attention kernels instead.  direct=True: the direct edge encoding
    (E[attn_edge_type] instead of the multi-hop walk; W gets no gradient)."""

    @staticmethod
    def forward(ctx, batch, R, Ppos, E, W, tvd, out_dtype, direct=False):
        Rc, Pc, Ec, Wc, tc = (t.detach().float().contiguous() for t in (R, Ppos, E, W, tvd))
        ctx.batch, ctx.num_bins, ctx.direct = batch, Ppos.shape[0], direct
        ctx.save_for_backward(Ec, Wc)
        return _bias_fwd(batch, direct, Rc, Pc, Ec, Wc, tc, out_dtype)

    @staticmethod
    def backward(ctx, dbias):
        E, W = ctx.saved_tensors
        dR, dP, dE, dW, dt = _bias_bwd(ctx.batch, ctx.direct, dbias.float().contiguous(), E, W, ctx.num_bins)
        return None, dR, dP, dE, dW, dt, None, None


# ----------------------------------------------------------------------------------------------- K3
SMALL_T = 16     # csrc/k3_small.cuh kSmallT: graphs of at most this many tokens take the SIMT attention kernels


def all_large(batch):
    """True when every graph of the batch has more than SMALL_T tokens (then the small-graph attention launch is skipped).
    A bucketed batch never claims it: its CUDA graph is replayed for other batches of the same bucket."""
    if getattr(batch, "padded", False) or getattr(batch, "n_host", None) is None or len(batch.n_host) == 0:
        return False
    return int(min(batch.n_host)) + 1 > SMALL_T


def _t_min(batch):
    """t_min_host of mobgt_attn_fwd / _bwd: the smallest token count of the batch, 0 = unknown (launch both kernels)."""
    return int(min(batch.n_host)) + 1 if all_large(batch) else 0


def _head_dim(qkv, H):
    """Head dim of a fused [ntok, 3*H*d] projection."""
    d, r = divmod(qkv.shape[1], 3 * H)
    assert r == 0, f"qkv width {qkv.shape[1]} is not 3 * H * d for H={H}"
    return d


def attn_fwd_raw(qkv, bias, batch, scale=None, drop_p=0.0, seed=0):
    """qkv bf16 [ntok, 3*H*d] (fused projection) ; bias bf16 [B,H,T,Tp] -> (out bf16 [ntok, H*d], lse f32 [ntok,H]).
    The head dim d comes from the qkv width (built: 16, 24); scale defaults to d ** -0.5.
    drop_p > 0: attention dropout on the probabilities (model_fqandtoyo.py:1704), mask = hash(seed, plane, row, col)."""
    ntok = qkv.shape[0]
    B, H, T, Tp = bias.shape
    hd = _head_dim(qkv, H)
    D = H * hd
    assert qkv.dtype == torch.bfloat16 and bias.dtype == torch.bfloat16 and qkv.is_contiguous()
    # a bucketed batch carries padding token rows no graph owns: the kernels never touch them, and they must hold finite values
    # (they flow through the row-wise layers and meet their zero gradients in the weight-gradient GEMMs)
    alloc = torch.zeros if getattr(batch, "padded", False) else torch.empty
    out = alloc(ntok, D, dtype=torch.bfloat16, device=qkv.device)
    lse = alloc(ntok, H, dtype=torch.float32, device=qkv.device)
    scale = float(hd ** -0.5) if scale is None else float(scale)
    base = qkv.data_ptr()
    _C.call("mobgt_attn_fwd_hd", base, base + 2 * D, base + 4 * D, 3 * D, _C.ptr(bias), _C.ptr(batch.tok_off), _C.ptr(getattr(batch, "size_order", None)), B, H,
            ntok, T, Tp, int(batch.N) + 1, _t_min(batch), scale, float(drop_p), int(seed), _C.ptr(_seed_dev) if drop_p > 0 else None, _C.ptr(out),
            _C.ptr(lse), hd, _C.stream_ptr())
    return out, lse


def attn_bwd_raw(qkv, bias, out, dout, lse, batch, dbias, accumulate, scale=None, drop_p=0.0, seed=0):
    """-> dqkv bf16 [ntok, 3*H*d]; dbias [B,H,T,Tp] is written in place: f32 overwritten (accumulate=0) / added to
    (accumulate=1), or bf16 overwritten (accumulate=2: this layer's own dS plane, TMA-stored)."""
    ntok = qkv.shape[0]
    B, H, T, Tp = bias.shape
    hd = _head_dim(qkv, H)
    D = H * hd
    assert dout.is_contiguous() and out.is_contiguous() and dbias.shape == bias.shape and dbias.is_contiguous()
    assert dbias.dtype == (torch.bfloat16 if accumulate == 2 else torch.float32)
    dqkv = torch.zeros_like(qkv) if getattr(batch, "padded", False) else torch.empty_like(qkv)    # padding rows: zero gradient
    scale = float(hd ** -0.5) if scale is None else float(scale)
    base, dbase = qkv.data_ptr(), dqkv.data_ptr()
    _C.call("mobgt_attn_bwd_hd", base, base + 2 * D, base + 4 * D, 3 * D, _C.ptr(bias), _C.ptr(out), _C.ptr(dout), _C.ptr(lse),
            _C.ptr(batch.tok_off), _C.ptr(getattr(batch, "size_order", None)), B, H, ntok, T, Tp, int(batch.N) + 1, _t_min(batch), scale, dbase, dbase + 2 * D, dbase + 4 * D, 3 * D,
            _C.ptr(dbias), int(accumulate), float(drop_p), int(seed), _C.ptr(_seed_dev) if drop_p > 0 else None, hd, _C.stream_ptr())
    return dqkv


class BiasedAttention(torch.autograd.Function):
    """softmax(scale * q k^T + bias) v per packed graph and head (model_fqandtoyo.py:1693-1706).

    The bias is ONE tensor used by every encoder layer.  Each layer's backward stores its own dS = d(bias) plane
    (bf16, written by a TMA store from the tile the dK / dQ MMAs consume) into bias_slot.planes[layer]; the gradient
    w.r.t. the bias tables is produced once, by BiasLink below, where mobgt_bias_bwd sums the planes in fp32."""

    @staticmethod
    def forward(ctx, qkv, bias_slot, layer, drop_p=0.0, scale=None):
        """drop_p: the attention dropout rate when training (`att_dropout`, model_fqandtoyo.py:1674, 1704), else 0.
        scale: MultiHeadAttention.scale (att_size ** -0.5); None: head dim ** -0.5."""
        seed = _next_drop_seed() if drop_p > 0 else 0
        out, lse = attn_fwd_raw(qkv, bias_slot.bias, bias_slot.batch, scale=scale, drop_p=drop_p, seed=seed)
        ctx.save_for_backward(qkv, out, lse)
        ctx.slot, ctx.layer, ctx.drop, ctx.scale = bias_slot, layer, (drop_p, seed), scale
        return out

    @staticmethod
    def backward(ctx, dout):
        qkv, out, lse = ctx.saved_tensors
        slot = ctx.slot
        if slot.planes is None:
            slot.planes = torch.empty((slot.n_layers,) + tuple(slot.bias.shape), dtype=torch.bfloat16, device=qkv.device)
            slot.written = set()
        dqkv = attn_bwd_raw(qkv, slot.bias, out, dout.contiguous(), lse, slot.batch, slot.planes[ctx.layer], 2, scale=ctx.scale,
                            drop_p=ctx.drop[0], seed=ctx.drop[1])
        slot.written.add(ctx.layer)
        return dqkv, None, None, None, None


def attn_f32_fwd_raw(qkv, bias, batch, scale=None, drop_p=0.0, seed=0):
    """fp32 mode of K3 (csrc/k3_attn_f32.cu): qkv f32 [ntok, 3*H*d], bias f32 [B,H,T,Tp] -> (out f32 [ntok, H*d], lse f32 [ntok,H])."""
    ntok = qkv.shape[0]
    B, H, T, Tp = bias.shape
    hd = _head_dim(qkv, H)
    D = H * hd
    assert qkv.dtype == torch.float32 and bias.dtype == torch.float32 and qkv.is_contiguous()
    alloc = torch.zeros if getattr(batch, "padded", False) else torch.empty
    out = alloc(ntok, D, dtype=torch.float32, device=qkv.device)
    lse = alloc(ntok, H, dtype=torch.float32, device=qkv.device)
    scale = float(hd ** -0.5) if scale is None else float(scale)
    base = qkv.data_ptr()
    _C.call("mobgt_attn_f32_fwd_hd", base, base + 4 * D, base + 8 * D, 3 * D, _C.ptr(bias), _C.ptr(batch.tok_off), B, H, ntok, T, Tp,
            int(batch.N) + 1, scale, float(drop_p), int(seed), _C.ptr(_seed_dev) if drop_p > 0 else None, _C.ptr(out), _C.ptr(lse),
            hd, _C.stream_ptr())
    return out, lse


def attn_f32_bwd_raw(qkv, bias, out, dout, lse, batch, dbias, accumulate, scale=None, drop_p=0.0, seed=0):
    """-> dqkv f32 [ntok, 3*H*d]; dbias f32 [B,H,T,Tp] overwritten (accumulate=0) or added to (accumulate=1), live cells only."""
    B, H, T, Tp = bias.shape
    hd = _head_dim(qkv, H)
    D = H * hd
    assert dout.is_contiguous() and out.is_contiguous() and dbias.shape == bias.shape and dbias.is_contiguous()
    assert dbias.dtype == torch.float32 and dout.dtype == torch.float32 and accumulate in (0, 1)
    dqkv = torch.zeros_like(qkv) if getattr(batch, "padded", False) else torch.empty_like(qkv)
    scale = float(hd ** -0.5) if scale is None else float(scale)
    base, dbase = qkv.data_ptr(), dqkv.data_ptr()
    _C.call("mobgt_attn_f32_bwd_hd", base, base + 4 * D, base + 8 * D, 3 * D, _C.ptr(bias), _C.ptr(out), _C.ptr(dout), _C.ptr(lse),
            _C.ptr(batch.tok_off), B, H, qkv.shape[0], T, Tp, int(batch.N) + 1, scale, dbase, dbase + 4 * D, dbase + 8 * D, 3 * D,
            _C.ptr(dbias), int(accumulate), float(drop_p), int(seed), _C.ptr(_seed_dev) if drop_p > 0 else None, hd, _C.stream_ptr())
    return dqkv


class BiasedAttentionF32(torch.autograd.Function):
    """BiasedAttention in fp32 mode (`Graphormer(precision=32)`): fp32 operands, bias and arithmetic.  The layers' dS are added
    into ONE fp32 [B,H,T,Tp] buffer (each cell has one writer per layer and the layers' backwards run one after the other, so the
    sum has a fixed order); BiasLink hands it to mobgt_bias_bwd."""

    @staticmethod
    def forward(ctx, qkv, bias_slot, layer, drop_p=0.0, scale=None):
        seed = _next_drop_seed() if drop_p > 0 else 0
        out, lse = attn_f32_fwd_raw(qkv, bias_slot.bias, bias_slot.batch, scale=scale, drop_p=drop_p, seed=seed)
        ctx.save_for_backward(qkv, out, lse)
        ctx.slot, ctx.layer, ctx.drop, ctx.scale = bias_slot, layer, (drop_p, seed), scale
        return out

    @staticmethod
    def backward(ctx, dout):
        qkv, out, lse = ctx.saved_tensors
        slot = ctx.slot
        if slot.planes is None:
            slot.planes = torch.zeros_like(slot.bias)
        dqkv = attn_f32_bwd_raw(qkv, slot.bias, out, dout.contiguous(), lse, slot.batch, slot.planes, 1, scale=ctx.scale,
                                drop_p=ctx.drop[0], seed=ctx.drop[1])
        slot.written.add(ctx.layer)
        return dqkv, None, None, None, None


class BiasSlot:
    """What the six encoder layers of one forward share: the batch, the bias tensor (written once by K2) and, in backward,
    the stack of per-layer bf16 dS planes (dtype bf16) or the one fp32 sum of the layers' dS (dtype fp32: precision=32)."""

    def __init__(self, batch, n_layers, bias=None, dtype=torch.bfloat16):
        self.bias, self.batch, self.n_layers, self.planes, self.written, self.dtype = bias, batch, n_layers, None, set(), dtype


class BiasLink(torch.autograd.Function):
    """The attention bias of a training forward as ONE autograd node on the token stream, in front of encoder layer 0.
    forward : K2 builds the bias from the five tables (model_fqandtoyo.py:1143-1216) into slot.bias — a plain tensor every
              layer's attention reads; the token tensor passes through unchanged (the input dropout site, :1347).
    backward: autograd reaches this node after EVERY layer's attention backward has stored its dS plane in slot.planes, so
              the table gradients are one K2-backward over the stack; d(tokens) passes through."""

    @staticmethod
    def forward(ctx, tok, slot, R, Ppos, E, W, tvd, direct=False):
        Rc, Pc, Ec, Wc, tc = (t.detach().float().contiguous() for t in (R, Ppos, E, W, tvd))
        slot.bias = _bias_fwd(slot.batch, direct, Rc, Pc, Ec, Wc, tc, slot.dtype)
        ctx.slot, ctx.num_bins, ctx.direct = slot, Ppos.shape[0], direct
        ctx.save_for_backward(Ec, Wc)
        return tok.view_as(tok)

    @staticmethod
    def backward(ctx, dtok):
        slot = ctx.slot
        planes, slot.planes = slot.planes, None
        if planes is None:                      # no attention layer took part in this backward
            return dtok, None, None, None, None, None, None, None
        if planes.dtype == torch.bfloat16:
            for l in range(slot.n_layers):      # a layer whose backward never ran contributes nothing
                if l not in slot.written:
                    planes[l].zero_()
        E, W = ctx.saved_tensors
        dR, dP, dE, dW, dt = _bias_bwd(slot.batch, ctx.direct, planes, E, W, ctx.num_bins)
        return dtok, None, dR, dP, dE, dW, dt, None


# ----------------------------------------------------------------------------------------------- K4
def embed_gather_raw(batch, cat_of_poi, Gd, Tm, Gc, out_dtype=torch.bfloat16):
    nn_ = int(batch.x_nodes.numel())
    Dp, Dt, Dc = Gd.shape[1], Tm.shape[1], Gc.shape[1]
    out = torch.empty(nn_, Dp + Dt + Dc, dtype=out_dtype, device=Gd.device)
    _C.call("mobgt_embed_gather_fwd", _C.ptr(batch.x_nodes), _C.ptr(batch.slot), _C.ptr(cat_of_poi), _C.ptr(Gd), _C.ptr(Tm),
            _C.ptr(Gc), nn_, Dp, Dt, Dc, _C.ptr(out), _dt(out), _C.stream_ptr())
    return out


def embed_sum_raw(batch, nf, Din, Dout, pe, graph_token):
    ntok = int(batch.tok_pos.numel())
    D = nf.shape[1]
    tok = torch.empty(ntok, D, dtype=nf.dtype, device=nf.device)
    _C.call("mobgt_embed_sum_fwd", _C.ptr(nf), _C.ptr(batch.tok_graph), _C.ptr(batch.tok_pos), _C.ptr(batch.in_deg),
            _C.ptr(batch.out_deg), _C.ptr(Din), _C.ptr(Dout), _C.ptr(pe), _C.ptr(graph_token), ntok, D, _C.ptr(tok), _dt(tok),
            _C.stream_ptr())
    return tok


def sort_plan(keys):
    """Stable sort of an int key stream -> (perm i32, keys_sorted i32): the fixed summation order of segment_sum."""
    ks, perm = torch.sort(keys.long(), stable=True)
    return perm.int().contiguous(), ks.int().contiguous()


def segment_sum_raw(src, col0, D, plan, nkeys, out=None):
    """table[key] = sum_{rows r: key_r == key} src[r, col0:col0+D]  (deterministic; fp32 out [nkeys, D])."""
    perm, ks = plan
    nrows = int(perm.numel())
    assert src.dim() == 2 and src.stride(1) == 1
    if out is None:
        out = torch.zeros(nkeys, D, dtype=torch.float32, device=src.device)
    nchunks = (nrows + 31) // 32
    ws_bytes = 2 * nchunks * D * 4 + 2 * nchunks * 4
    ws = torch.empty(max(ws_bytes, 16), dtype=torch.uint8, device=src.device)
    _C.call("mobgt_segment_sum", _C.ptr(src) if src.is_contiguous() else src.data_ptr(), _dt(src), src.stride(0), col0, D,
            _C.ptr(perm), _C.ptr(ks), nrows, _C.ptr(out), nkeys, _C.ptr(ws), ws_bytes, _C.stream_ptr())
    return out


class EmbedGather(torch.autograd.Function):
    """[Gd[x-1] | Tm[slot] | Gc[cat_of_poi[x-1]-1]] per packed node (model_fqandtoyo.py:1259-1264)."""

    @staticmethod
    def forward(ctx, batch, cat_of_poi, Gd, Tm, Gc, out_dtype, time_pad=None):
        """time_pad: padding_idx of the time-slot table (nn.Embedding(..., padding_idx=0) for foursquaregraph / gowalla,
        model_fqandtoyo.py:654, 796; None for toyotagraph, :915): that row receives no gradient."""
        ctx.batch, ctx.cat_of_poi, ctx.time_pad = batch, cat_of_poi, time_pad
        ctx.shapes = (Gd.shape, Tm.shape, Gc.shape)
        return embed_gather_raw(batch, cat_of_poi, Gd.detach().float().contiguous(), Tm.detach().float().contiguous(),
                                Gc.detach().float().contiguous(), out_dtype)

    @staticmethod
    def backward(ctx, dout):
        b = ctx.batch
        (P, Dp), (Tr, Dt), (C, Dc) = ctx.shapes
        dout = dout.contiguous()
        plans = b.__dict__.setdefault("_plans", {})
        if "poi" not in plans:
            b.build_plans()
        if "cat" not in plans:
            plans["cat"] = sort_plan(ctx.cat_of_poi[b.x_nodes.long() - 1].long() - 1)
        dGd = segment_sum_raw(dout, 0, Dp, plans["poi"], P)
        dTm = segment_sum_raw(dout, Dp, Dt, plans["slot"], Tr)
        dGc = segment_sum_raw(dout, Dp + Dt, Dc, plans["cat"], C)
        if ctx.time_pad is not None:
            dTm[ctx.time_pad].zero_()
        return None, None, dGd, dTm, dGc, None, None


class EmbedSum(torch.autograd.Function):
    """tokens = nf + in_degree_encoder + out_degree_encoder + pe[q+1] ; graph token + pe[0]
    (model_fqandtoyo.py:1288-1344).  Backward: d_nf = token-row gather; table grads by segment_sum."""

    @staticmethod
    def forward(ctx, batch, nf, Din, Dout, pe, graph_token):
        ctx.batch = batch
        ctx.shapes = (Din.shape, Dout.shape, pe.shape)
        return embed_sum_raw(batch, nf.contiguous(), Din.detach().float().contiguous(), Dout.detach().float().contiguous(),
                             pe.detach().float().contiguous(), graph_token.detach().float().contiguous().view(-1))

    @staticmethod
    def backward(ctx, dtok):
        b = ctx.batch
        dtok = dtok.contiguous()
        D = dtok.shape[1]
        plans = b.__dict__.setdefault("_plans", {})
        if "pos" not in plans:
            b.build_plans()
        (ri, _), (ro, _), (rp, _) = ctx.shapes
        d_nf = dtok.index_select(0, plans["node_rows"])
        dDin = segment_sum_raw(dtok, 0, D, plans["ind"], ri)
        dDout = segment_sum_raw(dtok, 0, D, plans["outd"], ro)
        dpe = segment_sum_raw(dtok, 0, D, plans["pos"], rp)
        dgt = dpe[0:1].clone()          # d graph_token = sum_g dtok[g, 0] = dpe[0]
        dDin[0].zero_()                 # padding_idx rows / graph-token rows carry key 0
        dDout[0].zero_()
        return None, d_nf, dDin, dDout, dpe, dgt



# ----------------------------------------------------------------------------------------------- K6
def colsum(src, out=None):
    """out[c] = sum_r src[r, c] in fp32 (src bf16 / f32 [N, C], last dim contiguous): the bias gradient of a Linear.
    out: optional f32 [C] destination (e.g. the parameter's slice of the flat gradient buffer)."""
    assert src.dim() == 2 and src.stride(1) == 1
    N, C = src.shape
    ws_bytes = int(_C.lib().mobgt_colsum_workspace_bytes(N, C))
    ws = torch.empty(max(ws_bytes, 16), dtype=torch.uint8, device=src.device)
    if out is None:
        out = torch.empty(C, dtype=torch.float32, device=src.device)
    _C.call("mobgt_colsum", src.data_ptr(), _dt(src), src.stride(0), N, C, _C.ptr(out), _C.ptr(ws), ws_bytes, _C.stream_ptr())
    return out


class LayerNormFn(torch.autograd.Function):
    """nn.LayerNorm over the last dim of a 2-D fp32 tensor (model_fqandtoyo.py:1731-1743, :1360-1364).  `want` selects the
    outputs: "f32", "bf16" (only the copy the next GEMM consumes) or "both" (residual stream + GEMM input); in backward the
    gradients of the two outputs are summed inside the kernel."""

    @staticmethod
    def forward(ctx, x, gamma, beta, eps, want):
        x = x.contiguous()
        N, D = x.shape
        dev = x.device
        out = torch.empty(N, D, dtype=torch.float32, device=dev)
        out16 = torch.empty(N, D, dtype=torch.bfloat16, device=dev) if want != "f32" else None
        mean = torch.empty(N, dtype=torch.float32, device=dev)
        rstd = torch.empty(N, dtype=torch.float32, device=dev)
        g, b = gamma.detach().float().contiguous(), beta.detach().float().contiguous()
        _C.call("mobgt_layernorm_fwd", _C.ptr(x), _C.ptr(g), _C.ptr(b), float(eps), N, D, _C.ptr(out), _C.ptr(out16), _C.ptr(mean),
                _C.ptr(rstd), _C.stream_ptr())
        ctx.save_for_backward(x, g, mean, rstd)
        ctx.want, ctx.masters = want, (gamma, beta)
        if want == "f32":
            return out
        if want == "bf16":
            return out16
        return out, out16

    @staticmethod
    def backward(ctx, *grads):
        x, g, mean, rstd = ctx.saved_tensors
        N, D = x.shape
        if ctx.want == "f32":
            dy32, dy16 = grads[0], None
        elif ctx.want == "bf16":
            dy32, dy16 = None, grads[0]
        else:
            dy32, dy16 = grads
        dy32 = dy32.contiguous() if dy32 is not None else None
        dy16 = dy16.contiguous() if dy16 is not None else None
        dx = torch.empty_like(x)
        tg, tb = _claim_vec(ctx.masters[0]), _claim_vec(ctx.masters[1])      # written in place when the flat buffer is fresh
        dgamma = tg if tg is not None else torch.empty(D, dtype=torch.float32, device=x.device)
        dbeta = tb if tb is not None else torch.empty(D, dtype=torch.float32, device=x.device)
        ws_bytes = int(_C.lib().mobgt_layernorm_bwd_workspace_bytes(D))
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=x.device)
        _C.call("mobgt_layernorm_bwd", _C.ptr(dy32), _C.ptr(dy16), _C.ptr(x), _C.ptr(g), _C.ptr(mean), _C.ptr(rstd), N, D, _C.ptr(dx),
                _C.ptr(dgamma), _C.ptr(dbeta), _C.ptr(ws), ws_bytes, _C.stream_ptr())
        return dx, (None if tg is not None else dgamma), (None if tb is not None else dbeta), None, None


def layer_norm(x, ln, want="f32"):
    """x f32 [N, D]; ln: an nn.LayerNorm (weight, bias, eps)."""
    return LayerNormFn.apply(x, ln.weight, ln.bias, ln.eps, want)


_drop_calls = 0
_seed_dev = None          # optional u64 device tensor folded into every dropout seed (CUDA-graph replays: graphs.GraphedTrainStep)


def set_device_seed(t):
    global _seed_dev
    _seed_dev = t


def _next_drop_seed():
    """A fresh 64-bit seed per dropout call, derived from torch's seed (torch.manual_seed makes runs reproducible)."""
    global _drop_calls
    _drop_calls += 1
    return (torch.initial_seed() * 0x9E3779B97F4A7C15 + _drop_calls * 0xD1B54A32D192ED03) & 0xFFFFFFFFFFFFFFFF


def _adln_fwd(x, y, gamma, beta, eps, p, want):
    """s = x + dropout(y) ; out = LayerNorm(s)  -> (s, out f32 | None, out bf16 | None, saved tensors, seed)"""
    x, y = x.contiguous(), y.contiguous()
    N, D = x.shape
    dev = x.device
    s = torch.empty(N, D, dtype=torch.float32, device=dev)
    out = torch.empty(N, D, dtype=torch.float32, device=dev) if want != "bf16" else None
    out16 = torch.empty(N, D, dtype=torch.bfloat16, device=dev) if want != "f32" else None
    mean = torch.empty(N, dtype=torch.float32, device=dev)
    rstd = torch.empty(N, dtype=torch.float32, device=dev)
    g, b = gamma.detach().float().contiguous(), beta.detach().float().contiguous()
    seed = _next_drop_seed() if p > 0 else 0
    _C.call("mobgt_add_dropout_layernorm_fwd", _C.ptr(x), _C.ptr(y), float(p), seed, _C.ptr(g), _C.ptr(b), float(eps), N, D,
            _C.ptr(s), _C.ptr(out), _C.ptr(out16), _C.ptr(mean), _C.ptr(rstd), _C.ptr(_seed_dev), _C.stream_ptr())
    return s, out, out16, (s, g, mean, rstd), seed


def _adln_bwd(saved, grads, p, seed, want, need_s, seed_dev, want_colsum=False, ln_masters=None, bias_masters=None):
    """-> (dx f32, dy bf16, dgamma, dbeta, column sums of dy | None).  ln_masters = (gamma, beta) / bias_masters = the bias
    parameter(s) of the Linear that produced y: when their gradient storage is fresh (`_claim`) the kernel writes dgamma / dbeta /
    the column sums straight into it and the corresponding return value is None."""
    s, g, mean, rstd = saved
    N, D = s.shape
    grads = list(grads)
    ds_ext = grads.pop(0) if need_s else None
    if want == "f32":
        dy32, dy16 = grads[0], None
    elif want == "bf16":
        dy32, dy16 = None, grads[0]
    else:
        dy32, dy16 = grads
    if dy32 is None and dy16 is None:          # only the residual branch carries a gradient
        dy32 = torch.zeros_like(s)
    c = lambda t: t.contiguous() if t is not None else None
    dy32, dy16, ds_ext = c(dy32), c(dy16), c(ds_ext)
    dx = torch.empty_like(s)
    dyb = torch.empty(N, D, dtype=torch.bfloat16, device=s.device)
    dgb = torch.empty(3 if want_colsum else 2, D, dtype=torch.float32, device=s.device)
    tg = _claim_vec(ln_masters[0]) if ln_masters is not None else None
    tb = _claim_vec(ln_masters[1]) if ln_masters is not None else None
    tc = _claim(bias_masters) if (bias_masters is not None and want_colsum) else None
    og, ob, oc = (tg if tg is not None else dgb[0]), (tb if tb is not None else dgb[1]), (tc if tc is not None else (dgb[2] if want_colsum else None))
    ws_bytes = int(_C.lib().mobgt_layernorm_bwd_workspace_bytes(D))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=s.device)
    _C.call("mobgt_add_dropout_layernorm_bwd", _C.ptr(dy32), _C.ptr(dy16), _C.ptr(ds_ext), _C.ptr(s), _C.ptr(g), _C.ptr(mean),
            _C.ptr(rstd), N, D, p, seed, _C.ptr(dx), _C.ptr(dyb), og.data_ptr(), ob.data_ptr(),
            oc.data_ptr() if want_colsum else None, _C.ptr(ws), ws_bytes, _C.ptr(seed_dev), _C.stream_ptr())
    return dx, dyb, (None if tg is not None else og), (None if tb is not None else ob), (_IN_PLACE if tc is not None else oc)


def _adln_outputs(s, out, out16, want, need_s):
    outs = {"f32": (out,), "bf16": (out16,), "both": (out, out16)}[want]
    return ((s,) + outs) if need_s else outs if len(outs) > 1 else outs[0]


class AddDropoutLayerNormFn(torch.autograd.Function):
    """The post-LN residual block of EncoderLayer.forward (model_fqandtoyo.py:1731-1743) in one kernel each way:
        s = x + dropout(y) ;  out = LayerNorm(s)
    x f32 [N, D] residual stream, y bf16 [N, D] sub-layer output.  Returns (s, outputs...) with outputs per `want` as in
    LayerNormFn; s is returned only when `need_s` (it feeds the next residual add)."""

    @staticmethod
    def forward(ctx, x, y, gamma, beta, eps, p, want, need_s):
        s, out, out16, saved, seed = _adln_fwd(x, y, gamma, beta, eps, p, want)
        ctx.save_for_backward(*saved)
        ctx.cfg = (float(p), seed, want, need_s)
        ctx.seed_dev, ctx.ln_masters = _seed_dev, (gamma, beta)
        return _adln_outputs(s, out, out16, want, need_s)

    @staticmethod
    def backward(ctx, *grads):
        p, seed, want, need_s = ctx.cfg
        dx, dyb, dgamma, dbeta, _ = _adln_bwd(ctx.saved_tensors, grads, p, seed, want, need_s, ctx.seed_dev, ln_masters=ctx.ln_masters)
        return dx, dyb, dgamma, dbeta, None, None, None, None


class LinearAddDropoutLNFn(torch.autograd.Function):
    """A sub-layer's closing Linear fused with the residual block that follows it (model_fqandtoyo.py:1708 + :1731-1735,
    :1655 + :1737-1741):   y = x16 W^T + b ;  s = resid + dropout(y) ;  out = LayerNorm(s).
    The GEMMs are the library's; fusing the two autograd nodes lets the LayerNorm-backward kernel hand the bias gradient of the
    Linear (the column sums of dy, accumulated while dy is written) straight to the parameter: no column-sum pass over dy."""

    @staticmethod
    def forward(ctx, x16, w16, b16, resid, gamma, beta, eps, p, want, need_s, *masters):
        y = torch.nn.functional.linear(x16, w16, b16)
        s, out, out16, saved, seed = _adln_fwd(resid, y, gamma, beta, eps, p, want)
        ctx.save_for_backward(x16, w16, *saved)
        ctx.cfg = (float(p), seed, want, need_s)
        ctx.seed_dev, ctx.masters, ctx.ln_masters = _seed_dev, masters, (gamma, beta)
        return _adln_outputs(s, out, out16, want, need_s)

    @staticmethod
    def backward(ctx, *grads):
        x16, w16 = ctx.saved_tensors[:2]
        p, seed, want, need_s = ctx.cfg
        m = len(ctx.masters) // 2
        dres, dy, dgamma, dbeta, dcol = _adln_bwd(ctx.saved_tensors[2:], grads, p, seed, want, need_s, ctx.seed_dev, want_colsum=True,
                                                  ln_masters=ctx.ln_masters, bias_masters=ctx.masters[m:])
        dx16 = dy @ w16
        pg = _deliver_param_grads(ctx.masters, dy.t(), x16, dcol)
        return (dx16, None, None, dres, dgamma, dbeta, None, None, None, None) + pg


# ----------------------------------------------------------------------------------------------- K10
def gemm_bf16(a, w, bias=None, mode=0, a2=None, w2=None, want_colsum=False, colsum_out=None):
    """C = epi(a w^T [, a2 w2^T], bias) on tcgen05 (csrc/k10_gemm.cu).  a bf16 [M, K], w bf16 [N, K] (nn.Linear layout), bias f32
    [N].  mode 0: + bias; 1: gelu(. + bias); 2: (a w^T) o gelu'(a2 w2^T + bias) [+ column sums].  -> C bf16 [M, N] (, colsum f32 [N])"""
    assert a.dtype == torch.bfloat16 and w.dtype == torch.bfloat16 and a.stride(1) == 1 and w.stride(1) == 1
    M, K = a.shape
    N = w.shape[0]
    C = torch.empty(M, N, dtype=torch.bfloat16, device=a.device)
    colsum, ws, nws = None, None, 0
    if mode == 2:
        assert a2 is not None and w2 is not None and a2.stride(1) == 1 and w2.stride(1) == 1
        if want_colsum:
            nws = int(_C.lib().mobgt_gemm_workspace_bytes(M, N, 2))
            ws = torch.empty(max(nws, 16), dtype=torch.uint8, device=a.device)
            colsum = colsum_out if colsum_out is not None else torch.empty(N, dtype=torch.float32, device=a.device)
    b = bias.detach().float().contiguous() if bias is not None else None
    _C.call("mobgt_gemm_bf16", a.data_ptr(), a.stride(0), w.data_ptr(), w.stride(0), _C.ptr(b), _C.ptr(C), N, M, N, K, int(mode),
            a2.data_ptr() if a2 is not None else None, a2.stride(0) if a2 is not None else 0,
            w2.data_ptr() if w2 is not None else None, w2.stride(0) if w2 is not None else 0,
            int(a2.shape[1]) if a2 is not None else 0, _C.ptr(colsum), _C.ptr(ws), nws, _C.stream_ptr())
    return (C, colsum) if mode == 2 else C


class FfnBlockFn(torch.autograd.Function):
    """FeedForwardNetwork + the residual block behind it (model_fqandtoyo.py:1644-1656, 1737-1741) as ONE autograd node:
        a = gelu(x W1^T + b1)            K10 mode 1: GEMM + bias + GELU in one kernel, the pre-activation never reaches HBM
        y = a W2^T + b2                  library GEMM (hidden output columns: 192 or 128)
        s = resid + dropout(y) ; out = LayerNorm(s)                                   K6
    backward:
        (dres, dy, dgamma, dbeta, db2)   K6 LayerNorm backward, db2 = column sums of dy from the same pass
        dh, db1 = (dy W2) o gelu'(x W1^T + b1), its column sums                       K10 mode 2 (pre-activation recomputed)
        dW2 = dy^T a ; dW1 = dh^T x ; dx = dh W1                                      library GEMMs (reductions over tokens)"""

    @staticmethod
    def forward(ctx, x16, w1, w2, b2, resid, gamma, beta, eps, p, want, need_s, m_w1, m_b1, m_w2, m_b2):
        a = gemm_bf16(x16, w1, m_b1, mode=1)
        y = torch.nn.functional.linear(a, w2, b2)            # N = encoder width (192, or 128 at hidden_dim 64): library GEMM
        s, out, out16, saved, seed = _adln_fwd(resid, y, gamma, beta, eps, p, want)
        ctx.save_for_backward(x16, w1, w2, a, *saved)
        ctx.cfg = (float(p), seed, want, need_s)
        ctx.seed_dev, ctx.masters, ctx.ln_masters = _seed_dev, (m_w1, m_b1, m_w2, m_b2), (gamma, beta)
        return _adln_outputs(s, out, out16, want, need_s)

    @staticmethod
    def backward(ctx, *grads):
        x16, w1, w2, a = ctx.saved_tensors[:4]
        p, seed, want, need_s = ctx.cfg
        m_w1, m_b1, m_w2, m_b2 = ctx.masters
        dres, dy, dgamma, dbeta, db2 = _adln_bwd(ctx.saved_tensors[4:], grads, p, seed, want, need_s, ctx.seed_dev, want_colsum=True,
                                                 ln_masters=ctx.ln_masters, bias_masters=(m_b2,))
        w2t = w2.t().contiguous()                                       # [ffn, hidden]: the B operand of dy W2
        t1 = _claim((m_b1,))
        dh, db1 = gemm_bf16(dy, w2t, m_b1, mode=2, a2=x16, w2=w1, want_colsum=True, colsum_out=t1)
        g_w2, g_b2 = _deliver_param_grads((m_w2, m_b2), dy.t(), a, db2)
        g_w1, g_b1 = _deliver_param_grads((m_w1, m_b1), dh.t(), x16, _IN_PLACE if t1 is not None else db1)
        dx16 = dh @ w1
        return (dx16, None, None, None, dres, dgamma, dbeta, None, None, None, None, g_w1, g_b1, g_w2, g_b2)


def ffn_block(x16, ffn, w1, w2, b2, resid, ln, p, training, want="f32", need_s=False):
    """LayerNorm(resid + dropout(ffn(x16))) with ffn = FeedForwardNetwork(layer1, GELU, layer2); w1 / w2 / b2: bf16 working
    copies (layer1's bias is applied in fp32 inside the K10 epilogue)."""
    if w1 is None:
        w1, w2 = ffn.layer1.weight.detach().to(torch.bfloat16), ffn.layer2.weight.detach().to(torch.bfloat16)
        b2 = ffn.layer2.bias.detach().to(torch.bfloat16)
    if w1.shape[0] % 128 != 0:
        raise NotImplementedError(f"ffn_dim={w1.shape[0]}: libmobgt's FFN kernels are built for multiples of 128")
    return FfnBlockFn.apply(x16, w1, w2, b2, resid, ln.weight, ln.bias, ln.eps, float(p) if training else 0.0, want, need_s,
                            ffn.layer1.weight, ffn.layer1.bias, ffn.layer2.weight, ffn.layer2.bias)


def linear_add_dropout_layer_norm(x16, lin, w16, b16, resid, ln, p, training, want="f32", need_s=False):
    """LayerNorm(resid + dropout(lin(x16)))  with lin's bf16 working copies w16 / b16 (None: cast on the fly)."""
    if w16 is None:
        w16, b16 = lin.weight.detach().to(torch.bfloat16), lin.bias.detach().to(torch.bfloat16)
    return LinearAddDropoutLNFn.apply(x16, w16, b16, resid, ln.weight, ln.bias, ln.eps, float(p) if training else 0.0, want, need_s,
                                      lin.weight, lin.bias)


def add_dropout_layer_norm(x, y, ln, p, training, want="f32", need_s=False):
    return AddDropoutLayerNormFn.apply(x, y, ln.weight, ln.bias, ln.eps, float(p) if training else 0.0, want, need_s)



_grad_ready = {}          # id(param) -> callable(param): fired when a Linear backward has finished that parameter's gradient


def on_grad_ready(param, fn):
    """Register `fn(param)` to run right after a libmobgt Linear backward has added `param`'s gradient into `param.grad` (the
    trainer starts the early all-reduce of out_proj.weight there).  fn=None removes the registration."""
    if fn is None:
        _grad_ready.pop(id(param), None)
    else:
        _grad_ready[id(param)] = fn


# ---- gradients written in place ------------------------------------------------------------------------------------------
# The trainer keeps every parameter gradient as a view of ONE flat fp32 buffer that it zeroes before each backward and tells
# this module about (`grads_zeroed`).  The FIRST gradient a parameter receives after that may simply be WRITTEN into its slice:
# the weight-gradient GEMM stores fp32 straight into the buffer (`torch.mm(..., out_dtype=float32, out=view)`: no bf16 rounding
# of dW, no cast, no add kernel) and the column-sum / LayerNorm-backward kernels get the slice as their output pointer.  A later
# gradient of the same parameter (a module applied twice, gradient accumulation without zeroing) is added, as autograd would.
_IN_PLACE = object()      # marker: "this gradient has already been written into the parameter's .grad"
_zero_epoch = 0
_zeroed_ranges = {}       # data_ptr of a zeroed flat buffer -> (lo, hi byte range, epoch of its last zeroing)
_last_written = {}        # id(param) -> epoch of its last in-place write


def grads_zeroed(flat):
    """The caller has just zeroed the flat gradient buffer `flat` (p.grad of its parameters are views of it)."""
    global _zero_epoch
    _zero_epoch += 1
    lo = flat.data_ptr()
    _zeroed_ranges[lo] = (lo, lo + flat.numel() * flat.element_size(), _zero_epoch)


def _claim(ps):
    """A writable fp32 tensor [sum of rows, ...] over the gradient storage of the parameters `ps` when (a) they own gradient
    views that lie back to back inside a flat buffer zeroed by `grads_zeroed` and (b) none of them has been written since that
    zeroing; else None (the caller then takes the accumulate path)."""
    if _zero_epoch == 0 or any(not (isinstance(p, torch.Tensor) and p.is_leaf) or p.grad is None for p in ps):
        return None
    g0 = ps[0].grad
    ptr = lo = g0.data_ptr()
    if lo % 16:           # (the kernels store with 128-bit accesses; optim.FlatAdamW / parallel.FlatGrads align every parameter)
        return None
    for p in ps:
        g = p.grad
        if g.dtype != torch.float32 or not g.is_contiguous() or g.data_ptr() != ptr or g.shape[1:] != g0.shape[1:]:
            return None
        ptr += g.numel() * 4
    epoch = max((e for a, b, e in _zeroed_ranges.values() if a <= lo and ptr <= b), default=0)
    if epoch == 0 or any(_last_written.get(id(p), -1) >= epoch for p in ps):
        return None
    for p in ps:
        _last_written[id(p)] = epoch
    if len(ps) == 1:
        return g0
    rows = sum(p.shape[0] for p in ps)
    shape = (rows,) + tuple(g0.shape[1:])
    stride, acc = [], 1
    for d in reversed(shape):
        stride.insert(0, acc)
        acc *= d
    return torch.as_strided(g0, shape, stride)


def _claim_vec(p):
    return _claim((p,))


def _deliver_param_grads(masters, at, bm, db):
    """Gradients of the fp32 master parameters of a (possibly fused) Linear: dW = at @ bm (at = dy^T [rows, tokens], bm = x
    [tokens, in], both bf16), db = the bias gradient f32 [rows] (or _IN_PLACE: a kernel has already written it).
    masters = (w_0, ..., w_{m-1}, b_0, ..., b_{m-1}).  With fresh flat gradient storage (`_claim`) dW is the fp32 output of the
    GEMM itself; with gradient views that have already been written it is added; without gradient buffers (plain autograd use)
    fp32 gradients are returned."""
    m = len(masters) // 2
    ws, bs = masters[:m], masters[m:]
    rows = [w.shape[0] for w in ws]
    tot = sum(rows)                           # (the working copy may carry zero padding rows behind the real ones)
    if all(p.grad is not None for p in masters):
        tw = _claim(ws)
        if tw is not None:
            torch.mm(at[:tot], bm, out_dtype=torch.float32, out=tw)
        else:
            dw16 = at @ bm
            r = 0
            for w in ws:
                w.grad.add_(dw16[r:r + w.shape[0]])
                r += w.shape[0]
        if db is not _IN_PLACE:
            tb = _claim(bs)
            if tb is not None:
                tb.copy_(db[:tot])
            else:
                r = 0
                for b in bs:
                    b.grad.add_(db[r:r + b.shape[0]])
                    r += b.shape[0]
        for w in ws:
            fn = _grad_ready.get(id(w))
            if fn is not None:
                fn(w)
        return (None,) * len(masters)
    dw = (at @ bm)[:tot].float()
    dbs = (None,) * m if db is _IN_PLACE else tuple(db[:tot].split(rows, 0))
    return tuple(dw.split(rows, 0)) + dbs


class LinearBiasFn(torch.autograd.Function):
    """y = x W^T + b with bf16 operands (library GEMMs).  w16 / b16 are the bf16 working copies of the fp32 master parameters
    `masters` = (w_0, ..., w_{m-1}, b_0, ..., b_{m-1}) — m > 1 when several nn.Linear are fused into one GEMM (q, k, v), their
    rows stacked in w16.  The gradients go straight to the masters in fp32 (`_deliver_param_grads`); the bias gradient
    dy.sum(0) is the K6 column-sum kernel (fp32 accumulation, fixed order) instead of torch's generic reduce."""

    @staticmethod
    def forward(ctx, x, w16, b16, *masters):
        ctx.save_for_backward(x, w16)
        ctx.masters = masters
        return torch.nn.functional.linear(x, w16, b16)

    @staticmethod
    def backward(ctx, dy):
        x, w16 = ctx.saved_tensors
        dy = dy.contiguous()
        dx = dy @ w16 if ctx.needs_input_grad[0] else None
        m = len(ctx.masters) // 2
        tot = sum(b.shape[0] for b in ctx.masters[m:])
        tb = _claim(ctx.masters[m:]) if tot == dy.shape[1] else None     # (a padded working copy: column sums via a temporary)
        db = colsum(dy, out=tb)
        grads = _deliver_param_grads(ctx.masters, dy.t(), x, _IN_PLACE if tb is not None else db)
        return (dx, None, None) + grads


_weight_epoch = 0


def weights_changed():
    """Called by an optimizer that writes parameters behind autograd's back (optim.FlatAdamW): invalidates every bf16
    working copy (Bf16Weights compares this counter next to the tensors' version counters)."""
    global _weight_epoch
    _weight_epoch += 1


class Bf16Weights:
    """bf16 working copies of a set of fp32 nn.Linear parameters, refreshed with ONE multi-tensor copy when an optimizer step
    has changed the masters (tensor version counters) — instead of a cast kernel + autograd node per parameter per step."""

    def __init__(self):
        self.groups = []          # (key, [linears])
        self.pad = {}
        self.bufs = {}
        self.stamp = None

    def register(self, key, linears, pad_rows_to=1):
        """pad_rows_to: round the row count of the working copy up to a multiple (zero rows / zero bias) — the head, whose
        class count (P + 1) is odd, is padded to a multiple of 8 so that its GEMMs and column sums stay 16-byte aligned."""
        self.groups.append((key, list(linears)))
        self.pad[key] = int(pad_rows_to)

    def _alloc(self, dev):
        for key, lins in self.groups:
            rows = sum(l.weight.shape[0] for l in lins)
            rows = (rows + self.pad[key] - 1) // self.pad[key] * self.pad[key]
            w = torch.zeros(rows, lins[0].weight.shape[1], dtype=torch.bfloat16, device=dev)
            b = torch.zeros(rows, dtype=torch.bfloat16, device=dev)
            self.bufs[key] = (w, b)
        self.dst, self.src = [], []
        for key, lins in self.groups:
            w, b = self.bufs[key]
            r = 0
            for l in lins:
                n = l.weight.shape[0]
                self.dst += [w[r:r + n], b[r:r + n]]
                self.src += [l.weight, l.bias]
                r += n

    def get(self, key):
        return self.bufs[key]

    def refresh(self):
        dev = self.groups[0][1][0].weight.device
        if not self.bufs or next(iter(self.bufs.values()))[0].device != dev:
            self._alloc(dev)
            self.stamp = None
        stamp = (sum(p._version for p in self.src), _weight_epoch)
        if stamp != self.stamp:
            with torch.no_grad():
                torch._foreach_copy_(self.dst, [p.detach() for p in self.src])
            self.stamp = (sum(p._version for p in self.src), _weight_epoch)


def linear_bf16(x, lin, w16=None, b16=None):
    """nn.Linear `lin` (fp32 master weights) applied to a bf16 [N, in] tensor; w16 / b16: its bf16 working copies."""
    if w16 is None:
        w16, b16 = lin.weight.detach().to(torch.bfloat16), lin.bias.detach().to(torch.bfloat16)
    return LinearBiasFn.apply(x, w16, b16, lin.weight, lin.bias)


def gelu_bwd_colsum_raw(da, h):
    """-> (dh bf16 [N, C] = da * gelu'(h), dbias f32 [C] = dh.sum(0)) in one pass."""
    assert da.dtype == torch.bfloat16 and h.dtype == torch.bfloat16 and da.is_contiguous() and h.is_contiguous() and da.shape == h.shape
    N, C = h.shape
    dh = torch.empty_like(h)
    db = torch.empty(C, dtype=torch.float32, device=h.device)
    ws_bytes = int(_C.lib().mobgt_colsum_workspace_bytes(N, C))
    ws = torch.empty(max(ws_bytes, 16), dtype=torch.uint8, device=h.device)
    _C.call("mobgt_gelu_bwd_colsum", _C.ptr(da), _C.ptr(h), N, C, _C.ptr(dh), _C.ptr(db), _C.ptr(ws), ws_bytes, _C.stream_ptr())
    return dh, db


class LinearGeluFn(torch.autograd.Function):
    """a = gelu(x W^T + b): FeedForwardNetwork.layer1 + nn.GELU (model_fqandtoyo.py:1646-1655) with bf16 operands.  The GEMM is
    the library's, and so is the forward GELU; in backward the activation gradient and the bias gradient (its column sum) come
    out of ONE pass over dA and h.  Gradients go straight to the fp32 master parameters."""

    @staticmethod
    def forward(ctx, x, w16, b16, w_master, b_master):
        h = torch.nn.functional.linear(x, w16, b16)
        ctx.save_for_backward(x, w16, h)
        ctx.masters = (w_master, b_master)
        return torch.nn.functional.gelu(h)

    @staticmethod
    def backward(ctx, da):
        x, w16, h = ctx.saved_tensors
        dh, db = gelu_bwd_colsum_raw(da.contiguous(), h)
        return (dh @ w16, None, None) + _deliver_param_grads(ctx.masters, dh.t(), x, db)


def linear_gelu_bf16(x, lin, w16=None, b16=None):
    """gelu(nn.Linear `lin`(x)) for a bf16 [N, in] tensor whose out_features is a multiple of 8."""
    if w16 is None:
        w16, b16 = lin.weight.detach().to(torch.bfloat16), lin.bias.detach().to(torch.bfloat16)
    return LinearGeluFn.apply(x, w16, b16, lin.weight, lin.bias)


class LinearF32BiasFn(torch.autograd.Function):
    """y = x W + b in fp32 storage (TF32 tensor cores when enabled): the dense half of a GraphConvolution whose output is wider
    than its input (modelGNN.py:39-46 associated as (adj x) W + b).  Same GEMMs as torch.addmm; the bias gradient — a sum over
    all P rows of the POI table — is the K6 column-sum kernel (fixed order) written straight into the parameter's gradient slice
    instead of torch's generic reduce (23 us per layer at P = 60 000)."""

    @staticmethod
    def forward(ctx, x, W, b):
        ctx.save_for_backward(x, W)
        ctx.bias = b
        return torch.addmm(b, x, W)

    @staticmethod
    def backward(ctx, dy):
        x, W = ctx.saved_tensors
        dy = dy.contiguous()
        dx = dy @ W.t() if ctx.needs_input_grad[0] else None
        dW = x.t() @ dy
        tb = _claim((ctx.bias,))
        db = colsum(dy, out=tb)
        return dx, dW, (None if tb is not None else db)


# ----------------------------------------------------------------------------------------------- K8
def spmm_csr_raw(csr, S, bias=None, slope=None):
    """Y = act(A @ S + bias): A = (crow i32 [n+1], col i32 [nnz], val f32 [nnz]); S f32 [m, D]; slope=None: no activation."""
    crow, col, val = csr
    n = int(crow.numel()) - 1
    S = S.contiguous()
    Y = torch.empty(n, S.shape[1], dtype=torch.float32, device=S.device)
    _C.call("mobgt_spmm_csr", _C.ptr(crow), _C.ptr(col), _C.ptr(val), n, _C.ptr(S), int(S.shape[1]), _C.ptr(bias),
            float(slope if slope is not None else 0.0), 0 if slope is None else 1, _C.ptr(Y), _C.stream_ptr())
    return Y


class SpmmFn(torch.autograd.Function):
    """Y = act(A @ S + bias) for a constant sparse A (the row-normalised adjacency of a global GCN, modelGNN.py:39-46).
    Backward: g = dY * act'(Y);  dS = A^T @ g (the same kernel on the CSR of A^T);  dbias = column sum of g (K6)."""

    @staticmethod
    def forward(ctx, A, At, S, bias, slope):
        b = bias.detach().float().contiguous() if bias is not None else None
        Y = spmm_csr_raw(A, S.detach().float(), b, slope)
        ctx.At, ctx.slope, ctx.has_bias, ctx.bias = At, slope, bias is not None, bias
        if slope is not None:
            ctx.save_for_backward(Y)
        return Y

    @staticmethod
    def backward(ctx, dY):
        g = dY.contiguous()
        if ctx.slope is not None:
            (Y,) = ctx.saved_tensors
            g = torch.ops.aten.leaky_relu_backward(g, Y, float(ctx.slope), True)     # one kernel (sign taken from the output)
        At = ctx.At
        if len(At) == 2:          # (chunked A^T, fold): long rows of A^T were cut into chunks, summed by a second tiny SpMM
            dS = spmm_csr_raw(At[1], spmm_csr_raw(At[0], g))
        else:
            dS = spmm_csr_raw(At, g)
        db = None
        if ctx.has_bias:
            tb = _claim((ctx.bias,))
            db = colsum(g, out=tb)
            if tb is not None:
                db = None
        return None, None, dS, db, None


def spmm(A, At, S, bias=None, slope=None):
    return SpmmFn.apply(A, At, S, bias, slope)


# ----------------------------------------------------------------------------------------------- K7
def enable_tf32(on=True):
    """The few GEMMs that stay in fp32 storage (GCN dense parts modelGNN.py:39, user fuse, cat_decoder, out_proj) run on the
    TF32 tensor cores.  This is cuBLAS's process-wide switch: it is set once, when a model asks for it (Graphormer(tf32=True);
    Graphormer(precision=32) and tf32=False ask for IEEE fp32 instead), not inside forward."""
    torch.backends.cuda.matmul.allow_tf32 = bool(on)


def _loss_ws(B, V, dev):
    n = int(_C.lib().mobgt_loss_workspace_bytes(B, V))
    if n < 0:
        raise _C.MobgtError(f"mobgt_loss_workspace_bytes rejected B={B} V={V}")
    return torch.empty(max(n, 16), dtype=torch.uint8, device=dev), n


class LogSoftmaxNllFn(torch.autograd.Function):
    """mean_{rows: target != ignore_index} -log_softmax(logits)[target]  (model_fqandtoyo.py:1425, 1470-1471; data.py:165)."""

    @staticmethod
    def forward(ctx, logits, target, ignore_index, n_classes=None):
        assert logits.dim() == 2 and logits.is_contiguous()
        B, Vp = logits.shape
        V = int(n_classes) if n_classes is not None else Vp          # columns [V, Vp) are row padding: not classes
        assert V <= Vp < V + 16
        target = target.contiguous().long()
        ws, nws = _loss_ws(B, V, logits.device)
        lse = torch.empty(B, dtype=torch.float32, device=logits.device)
        loss = torch.empty(2, dtype=torch.float32, device=logits.device)
        _C.call("mobgt_lsm_nll_fwd", logits.data_ptr(), _dt(logits), Vp, _C.ptr(target), int(ignore_index), B, V,
                _C.ptr(ws), nws, _C.ptr(lse), _C.ptr(loss), _C.stream_ptr())
        ctx.save_for_backward(logits, target, lse, loss)
        ctx.ignore_index, ctx.V = int(ignore_index), V
        return loss[0]

    @staticmethod
    def backward(ctx, g):
        logits, target, lse, loss = ctx.saved_tensors
        B, Vp = logits.shape
        g = g.detach().float().contiguous().view(1)
        dl = torch.empty(B, Vp, dtype=logits.dtype, device=logits.device)
        _C.call("mobgt_lsm_nll_bwd", logits.data_ptr(), _dt(logits), Vp, _C.ptr(target), ctx.ignore_index, B, ctx.V,
                _C.ptr(lse), _C.ptr(loss), _C.ptr(g), _C.ptr(dl), Vp, _C.stream_ptr())
        return dl, None, None, None


def log_softmax_nll_loss(logits, target, ignore_index=0, n_classes=None):
    """n_classes < logits.shape[1]: the trailing columns are row padding (not classes)."""
    return LogSoftmaxNllFn.apply(logits, target, ignore_index, n_classes)


class GradientTailLossFn(torch.autograd.Function):
    """GradientTailLoss(inputs, targets, alpha) with beta = k = 1 (model_fqandtoyo.py:545-550)."""

    @staticmethod
    def forward(ctx, logits, target, alpha, n_classes=None):
        assert logits.dim() == 2 and logits.is_contiguous()
        B, Vp = logits.shape
        V = int(n_classes) if n_classes is not None else Vp
        assert V <= Vp < V + 16
        target = target[:B].contiguous().long()              # :547 `targets[:len(inputs)]`
        ws, nws = _loss_ws(B, V, logits.device)
        loss = torch.empty(1, dtype=torch.float32, device=logits.device)
        _C.call("mobgt_gtl_fwd", logits.data_ptr(), _dt(logits), Vp, _C.ptr(target), float(alpha), B, V, _C.ptr(ws),
                nws, _C.ptr(loss), _C.stream_ptr())
        ctx.save_for_backward(logits, target)
        ctx.alpha, ctx.V = float(alpha), V
        return loss[0]

    @staticmethod
    def backward(ctx, g):
        logits, target = ctx.saved_tensors
        B, Vp = logits.shape
        g = g.detach().float().contiguous().view(1)
        dl = torch.empty(B, Vp, dtype=logits.dtype, device=logits.device)
        _C.call("mobgt_gtl_bwd", logits.data_ptr(), _dt(logits), Vp, _C.ptr(target), ctx.alpha, B, ctx.V, _C.ptr(g),
                _C.ptr(dl), Vp, _C.stream_ptr())
        return dl, None, None, None


def gradient_tail_loss(logits, target, alpha=0.25, n_classes=None):
    return GradientTailLossFn.apply(logits, target, alpha, n_classes)


# ----------------------------------------------------------------------------------------------- K5
def head_split(M, V, dtype=torch.bfloat16):
    """Number of per-row output lists = 2 x (vocabulary splits per 128-row tile of z): every CTA of mobgt_head_topk runs two
    epilogue groups.  The split count minimises waves x (tiles per CTA + a fixed per-CTA cost) over the 148 SMs.  (Measured on
    B200, c5 shard: 9 splits x 32 row tiles in two waves (573 us) beat 4 splits in one 86 %-full wave (638 us): the warm-up
    of a fresh top-k list costs ~8 tiles once the lists of a row share their pruning bound.)
    dtype=torch.float32: the split rule of mobgt_head_topk_f32 (`_head_split_f32`)."""
    if dtype == torch.float32:
        return _head_split_f32(M, V)
    mt = (M + 127) // 128
    nt = (V + 255) // 256          # vocabulary tiles of 256 rows (csrc/k5_head.cu kNT)
    best, best_cost = 1, None
    for gs in range(1, min(80, nt) + 1):
        waves = (mt * gs + 147) // 148
        cost = waves * ((nt + gs - 1) // gs + 4)
        if best_cost is None or cost < best_cost:
            best, best_cost = gs, cost
    return 2 * best


def _head_split_f32(M, V):
    """Lists per row of mobgt_head_topk_f32 = 4 x (vocabulary splits per 64-row tile of z): four scanner threads per row in
    every CTA.  Same cost model as the bf16 head (waves x (128-column tiles per CTA + a fixed cost)), one CTA per SM, at most
    40 splits so that the merge sees at most 160 lists."""
    mt = (M + 63) // 64
    nt = (V + 127) // 128          # vocabulary tiles of 128 rows (csrc/k5_head_f32.cu kBN)
    best, best_cost = 1, None
    for gs in range(1, min(40, nt) + 1):
        waves = (mt * gs + 147) // 148
        cost = waves * ((nt + gs - 1) // gs + 2)
        if best_cost is None or cost < best_cost:
            best, best_cost = gs, cost
    return 4 * best


def _head_entry(z, W):
    """The K5 entry point for z's dtype: float32 -> mobgt_head_topk_f32 (IEEE fp32 on the CUDA cores, W float32 too: it is
    never rounded here), anything else -> mobgt_head_topk (bf16 operands on tcgen05)."""
    if z.dtype != torch.float32:
        return "mobgt_head_topk"
    if W.dtype != torch.float32:
        raise TypeError(f"fp32 K5 head: W must be float32 like z, got {W.dtype}")
    return "mobgt_head_topk_f32"


def head_topk_local(z, W, bias, target, k, vocab_offset=0, st=None, dump_logits=False, nsplit=None):
    """One vocabulary shard.  z [M,K] and W [V,K] both bf16 (tcgen05 head) or both float32 (fp32 head), bias f32 [V]|None,
    target i32 [M] (global ids).  st=None -> runs mode 0 first (single-shard use).  nsplit: lists per row (default
    head_split; the merged result does not depend on it).  Returns dict(val [M,k], idx [M,k], cnt [M] (partial rank), st)."""
    M, K = z.shape
    V = W.shape[0]
    dev = z.device
    fn = _head_entry(z, W)
    ns = head_split(M, V, z.dtype) if nsplit is None else nsplit
    s = _C.stream_ptr()
    args = (_C.ptr(z), _C.ptr(W), _C.ptr(bias), _C.ptr(target), M, V, K, int(vocab_offset), k, ns)
    if st is None:
        st = torch.full((M,), float("-inf"), dtype=torch.float32, device=dev)
        _C.call(fn, *args, 0, _C.ptr(st), None, None, None, None, None, None, s)
    tv = torch.empty(M, ns, k, dtype=torch.float32, device=dev)
    ti = torch.empty(M, ns, k, dtype=torch.int32, device=dev)
    cg = torch.empty(M, ns, dtype=torch.int32, device=dev)
    ce = torch.empty(M, ns, dtype=torch.int32, device=dev)
    logits = torch.empty(M, V, dtype=torch.float32, device=dev) if dump_logits else None
    # per-row pruning bound shared by all lists of the row (the fp32 head keeps its lists independent and takes none)
    share = torch.zeros(M, dtype=torch.int32, device=dev) if fn == "mobgt_head_topk" else None
    _C.call(fn, *args, 1, _C.ptr(st), _C.ptr(tv), _C.ptr(ti), _C.ptr(cg), _C.ptr(ce), _C.ptr(logits), _C.ptr(share), s)
    val = torch.empty(M, k, dtype=torch.float32, device=dev)
    idx = torch.empty(M, k, dtype=torch.int32, device=dev)
    cnt = torch.empty(M, dtype=torch.int32, device=dev)
    _C.call("mobgt_topk_merge", _C.ptr(tv), _C.ptr(ti), _C.ptr(cg), _C.ptr(ce), M, ns, k, _C.ptr(val), _C.ptr(idx), _C.ptr(cnt), s)
    return dict(val=val, idx=idx, cnt=cnt, st=st, logits=logits)


def head_target_logit(z, W, bias, target, vocab_offset=0):
    """mode 0 only: st[row] = target logit if this shard owns the target, else -inf.  bf16 or float32 operands, as
    head_topk_local."""
    M, K = z.shape
    V = W.shape[0]
    st = torch.full((M,), float("-inf"), dtype=torch.float32, device=z.device)
    fn = _head_entry(z, W)
    _C.call(fn, _C.ptr(z), _C.ptr(W), _C.ptr(bias), _C.ptr(target), M, V, K, int(vocab_offset), 1,
            2 if fn == "mobgt_head_topk" else 4, 0, _C.ptr(st), None, None, None, None, None, None, _C.stream_ptr())
    return st


def topk_merge_lists(val, idx):
    """val/idx [M, S, k] (each list sorted) -> merged [M, k]."""
    M, S, k = val.shape
    ov = torch.empty(M, k, dtype=torch.float32, device=val.device)
    oi = torch.empty(M, k, dtype=torch.int32, device=val.device)
    _C.call("mobgt_topk_merge", _C.ptr(val.contiguous()), _C.ptr(idx.contiguous()), None, None, M, S, k, _C.ptr(ov), _C.ptr(oi),
            None, _C.stream_ptr())
    return ov, oi


def head_topk_sharded(z, W_shard, bias_shard, target, k, vocab_offset, group=None):
    """Vocabulary-parallel evaluation head (SURVEY.md §8e): every rank holds rows [vocab_offset, vocab_offset+V_r) of
    out_proj and the full z.  The collective choreography (s_t all-reduce MAX -> local top-k / counts -> all-gather of the
    lists over NVLink -> all-reduce SUM of the counts -> k-way merge, ties -> lower index) lives in parallel.py so that it
    is also exercised over gloo on CPU; here it is bound to the libmobgt kernels."""
    import sys
    from . import parallel
    return parallel.sharded_head_topk(sys.modules[__name__], z, W_shard, bias_shard, target, k, vocab_offset, group)


def metrics_from_rank(rank, target, ks=(1, 5, 10, 20)):
    """Acc@k / NDCG@k / MRR sums from the 0-based rank of each target (== the reference's get_acc / MRR_metric sums,
    model_fqandtoyo.py:48-90, 122-131, including `target > 0` and the break at the first target == 0)."""
    r = rank.double()
    t = target.view(-1)
    zero = (t == 0).nonzero()
    stop = int(zero[0]) if len(zero) else len(t)
    live = torch.zeros_like(t, dtype=torch.bool)
    live[:stop] = True
    out = {}
    for k in ks:
        hit = live & (rank < k) & (t > 0)
        out[f"acc{k}"] = float(hit.sum())
        out[f"ndcg{k}"] = float((1.0 / torch.log2(r[hit] + 2)).sum())
    out["mrr"] = float((1.0 / (r + 1)).sum())
    return out
