"""`Graphormer` — the MobGT network (reference: graphormer/model_fqandtoyo.py:580-1641), B200-native hot path.

Drop-in surface kept from the reference:
  * constructor hyper-parameters / flag names (model_fqandtoyo.py:581-603, 1619-1641, incl. the reference's own
    spelling `intput_dropout_rate`);
  * `forward(batched_data, perturb=None) -> [poi_logits, cat_logits]` (:1123, :1393-1428);
  * `training_step`, `validation_step`, `test_step`, `test_epoch_end`, `configure_optimizers` (:1434-1616);
  * parameter names (`state_dict` keys) of every module the live forward uses.
The reference's host loops (per-graph embedding loop :1257-1269, per-token user fuse :1353-1358 — of which only token 0 is
ever consumed, :1394-1396) are replaced by packed var-len tensors and the libmobgt kernels:
  K2 AttnBias -> K4 EmbedGather / EmbedSum -> 6 x (fused QKV GEMM -> K3 BiasedAttention -> FFN) -> user fuse -> heads.
Padding tokens are never materialised: their keys are masked (-inf columns) in every layer and only token 0 reaches
the heads, so logits and all gradients are identical to the padded computation.
"""
import math

import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional as F

from . import ops
from .lr import PolynomialDecayLR

NODE_DIM = 2000    # model_fqandtoyo.py:567
# (num_heads, hidden_dim) pairs the kernels are built for: K2 is built for 8 and 12 heads, K3 for head dims
# (hidden_dim + 64) / num_heads = 16, 24.  Each pair also fixes the final LayerNorm / K5 head width 2 * hidden_dim + 64.
SUPPORTED_SHAPES = frozenset({(8, 64), (8, 128), (12, 128)})

DATASET_TRAITS = {
    # per-dataset constructor differences (model_fqandtoyo.py:636-779, 781-900, 902-1029)
    "foursquaregraph": dict(time_rows=49, time_pad=0, user_extra=0, cat_extra=0, poi_extra=0, log_softmax=False),
    "gowalla_nevda": dict(time_rows=48, time_pad=0, user_extra=0, cat_extra=1, poi_extra=1, log_softmax=False),
    "gowalla_7day": dict(time_rows=48, time_pad=0, user_extra=0, cat_extra=1, poi_extra=1, log_softmax=False),
    "toyotagraph": dict(time_rows=48, time_pad=None, user_extra=1, cat_extra=0, poi_extra=1, log_softmax=True),
}


def _csr_transpose(csr, n, ncols=None):
    """CSR (crow, col, val) of the transpose of an n x ncols CSR matrix (numpy, stable: rows of A^T keep ascending columns)."""
    ncols = n if ncols is None else ncols
    crow, col, val = (np.asarray(a) for a in csr)
    rows = np.repeat(np.arange(n), np.diff(crow))
    order = np.argsort(col, kind="stable")
    tcrow = np.zeros(ncols + 1, np.int64)
    np.cumsum(np.bincount(col, minlength=ncols), out=tcrow[1:])
    return tcrow, rows[order], np.asarray(val)[order]


def _csr_split_rows(csr, chunk=128):
    """Cut the rows of a CSR matrix into chunks of <= `chunk` non-zeros -> (chunked CSR, fold CSR): the chunked matrix has one
    row per chunk (K8 is row-parallel: a 60 000-entry row of a transposed feature matrix would serialise one sub-warp), the
    fold matrix [rows, chunks] of ones adds the chunks of every original row back together (a second K8 call, fixed order)."""
    crow, col, val = (np.asarray(a) for a in csr)
    n = len(crow) - 1
    starts, owner = [], []
    for r in range(n):
        a, b = int(crow[r]), int(crow[r + 1])
        for s0 in range(a, max(b, a + 1), chunk):
            starts.append(min(s0, b))
            owner.append(r)
    vcrow = np.array(starts + [int(crow[-1])], np.int64)
    owner = np.array(owner, np.int64)
    fcrow = np.zeros(n + 1, np.int64)
    np.cumsum(np.bincount(owner, minlength=n), out=fcrow[1:])
    return (vcrow, col, val), (fcrow, np.arange(len(owner), dtype=np.int64), np.ones(len(owner), np.float32))


def _dense_to_csr(d):
    rows, cols = np.nonzero(d)
    crow = np.zeros(d.shape[0] + 1, np.int64)
    np.cumsum(np.bincount(rows, minlength=d.shape[0]), out=crow[1:])
    return crow, cols.astype(np.int64), d[rows, cols].astype(np.float32)


class GraphConvolution(nn.Module):
    """modelGNN.py:21-50: `adj @ (x @ W) + b`.  The sparse product is K8 (ops.spmm, csrc/k8_spmm.cu).  It is associated so that
    the gather runs at the NARROWER of the two widths: out <= in -> `adj @ (x W)` with bias (and the following LeakyReLU)
    fused into the SpMM store; out > in -> `(adj @ x) W + b` (the dense part is a library GEMM either way)."""

    def __init__(self, in_features, out_features):
        super().__init__()
        self.weight = nn.Parameter(torch.empty(in_features, out_features))
        self.bias = nn.Parameter(torch.empty(out_features))
        stdv = 1.0 / math.sqrt(out_features)
        self.weight.data.uniform_(-stdv, stdv)
        self.bias.data.uniform_(-stdv, stdv)

    def forward(self, x, adj, slope=None, x_csr=None):
        """adj = (A, At): CSR triples (crow, col, val) of the row-normalised adjacency and of its transpose.
        slope: fuse LeakyReLU(slope) of GCN.forward (modelGNN.py:67-69) into this layer.
        x_csr = (X, Xt): the layer INPUT as CSR triples, when it is a sparse constant of the dataset (the POI feature matrix:
        check-in frequency, one-hot category, lat, lon — 4 non-zeros in 3 + C columns, model_fqandtoyo.py:816-832): `x @ W`
        and its weight gradient `x^T dY` are then K8 gathers instead of dense GEMMs that stream the [P, 3 + C] fp32 matrix."""
        A, At = adj
        fin, fout = self.weight.shape
        ok = (16, 32, 64, 128)                                       # the widths K8 is built for
        if fout in ok and (fout <= fin or fin not in ok):
            xw = ops.spmm(x_csr[0], x_csr[1], self.weight) if x_csr is not None else torch.mm(x, self.weight)
            return ops.spmm(A, At, xw, self.bias, slope)
        if fin in ok:
            y = ops.LinearF32BiasFn.apply(ops.spmm(A, At, x), self.weight, self.bias)
            return F.leaky_relu(y, slope) if slope is not None else y
        raise NotImplementedError(f"GraphConvolution {fin}->{fout}: libmobgt's SpMM is built for widths 16 / 32 / 64 / 128")


class GCN(nn.Module):
    """modelGNN.py:53-73"""

    def __init__(self, ninput, nhid, noutput, dropout):
        super().__init__()
        ch = [ninput] + nhid + [noutput]
        self.gcn = nn.ModuleList([GraphConvolution(ch[i], ch[i + 1]) for i in range(len(ch) - 1)])
        self.dropout = dropout

    def forward(self, x, adj, x_csr=None):
        for i in range(len(self.gcn) - 1):
            x = self.gcn[i](x, adj, slope=0.2, x_csr=x_csr if i == 0 else None)   # F.leaky_relu(self.gcn[i](x, adj), 0.2)
        x = F.dropout(x, self.dropout, training=self.training)
        return self.gcn[-1](x, adj)


class FuseEmbeddings(nn.Module):
    """model_fqandtoyo.py:440-455"""

    def __init__(self, d1, d2):
        super().__init__()
        self.fuse_embed = nn.Linear(d1 + d2, d1 + d2)

    def forward(self, a, b):
        return F.leaky_relu(self.fuse_embed(torch.cat((a, b), a.dim() - 1)), 0.2)


class UserEmbeddings(nn.Module):
    """model_fqandtoyo.py:411-422"""

    def __init__(self, n, d):
        super().__init__()
        self.user_embedding = nn.Embedding(n, d)

    def forward(self, i):
        return self.user_embedding(i)


class LearnablePositionalEncoding(nn.Module):
    """model_fqandtoyo.py:330-358: pe[q+1] is added to node q ('node_reverse'), pe[0] to the graph token ('pos0');
    both are fused into K4 (ops.EmbedSum); this module only owns the table (and the reference's Dropout(0.1))."""

    def __init__(self, d_model, max_len, dropout=0.1):
        super().__init__()
        self.pe = nn.Parameter(torch.empty(d_model, max_len))
        nn.init.uniform_(self.pe, -0.02, 0.02)
        self.p = dropout


class FeedForwardNetwork(nn.Module):
    """model_fqandtoyo.py:1644-1656"""

    def __init__(self, hidden_size, ffn_size, dropout_rate):
        super().__init__()
        self.layer1 = nn.Linear(hidden_size, ffn_size)
        self.gelu = nn.GELU()
        self.layer2 = nn.Linear(ffn_size, hidden_size)

    def forward(self, x):
        return self.layer2(self.gelu(self.layer1(x)))


class MultiHeadAttention(nn.Module):
    """model_fqandtoyo.py:1659-1711.  q/k/v projections run as ONE fused GEMM (their weights stay separate parameters
    for state_dict compatibility); the core softmax(q k^T * scale + bias) v is K3 (ops.BiasedAttention)."""

    def __init__(self, hidden_size, attention_dropout_rate, num_heads):
        super().__init__()
        self.num_heads = num_heads
        self.att_size = hidden_size // num_heads
        self.scale = self.att_size ** -0.5
        self.linear_q = nn.Linear(hidden_size, num_heads * self.att_size)
        self.linear_k = nn.Linear(hidden_size, num_heads * self.att_size)
        self.linear_v = nn.Linear(hidden_size, num_heads * self.att_size)
        self.attention_dropout_rate = attention_dropout_rate
        self.output_layer = nn.Linear(num_heads * self.att_size, hidden_size)

    def forward(self, x16, bias_slot, layer=0, w16=None):
        """x16: bf16 [ntok, hidden] (the LayerNorm kernel of the previous layer emits this copy); w16: Bf16Weights or None."""
        q, k, v = self.linear_q, self.linear_k, self.linear_v
        if w16 is not None:
            wq, bq = w16.get((layer, "qkv"))
            wo, bo = w16.get((layer, "o"))
        else:
            wq = torch.cat([q.weight, k.weight, v.weight], 0).detach().to(torch.bfloat16)
            bq = torch.cat([q.bias, k.bias, v.bias], 0).detach().to(torch.bfloat16)
            wo = bo = None
        qkv = ops.LinearBiasFn.apply(x16, wq, bq, q.weight, k.weight, v.weight, q.bias, k.bias, v.bias)
        # attention output BEFORE output_layer: the caller fuses that Linear with the residual block (ops.LinearAddDropoutLNFn)
        return ops.BiasedAttention.apply(qkv, bias_slot, layer, self.attention_dropout_rate if self.training else 0.0,
                                         self.scale), wo, bo   # :1704


class EncoderLayer(nn.Module):
    """model_fqandtoyo.py:1714-1743 (post-LN variant of the live model; `self_attention_norm` exists but is unused)."""

    def __init__(self, hidden_size, ffn_size, dropout_rate, attention_dropout_rate, num_heads):
        super().__init__()
        self.self_attention_norm = nn.LayerNorm(hidden_size)
        self.self_attention = MultiHeadAttention(hidden_size, attention_dropout_rate, num_heads)
        self.self_attention_dropout = nn.Dropout(dropout_rate)
        self.ffn_norm1 = nn.LayerNorm(hidden_size)
        self.ffn_norm2 = nn.LayerNorm(hidden_size)
        self.ffn = FeedForwardNetwork(hidden_size, ffn_size, dropout_rate)
        self.ffn_dropout = nn.Dropout(dropout_rate)

    def forward(self, x, x16, bias_slot, layer=0, w16=None):
        """x: fp32 residual stream [ntok, hidden]; x16: its bf16 copy.  Residual stream and LayerNorms in fp32, GEMMs /
        attention in bf16 (the reference's --precision 16 AMP split).  Each residual add + dropout + LayerNorm is one K6 kernel
        per direction; the Linear bias gradients are the K6 column sum."""
        a, wo, bo = self.self_attention(x16, bias_slot, layer, w16)
        x1, y16 = ops.linear_add_dropout_layer_norm(a, self.self_attention.output_layer, wo, bo, x, self.ffn_norm1,
                                                    self.self_attention_dropout.p, self.training, "bf16", need_s=True)   # :1708, :1731-1735
        w1 = w16.get((layer, "f1"))[0] if w16 is not None else None
        w2, b2 = w16.get((layer, "f2")) if w16 is not None else (None, None)
        return ops.ffn_block(y16, self.ffn, w1, w2, b2, x1, self.ffn_norm2, self.ffn_dropout.p, self.training, "both")   # :1644-1656, :1737-1741

    def forward_f32(self, x, bias_slot, layer=0):
        """precision=32: the same layer with fp32 operands everywhere (IEEE fp32 GEMMs, the fp32 attention kernels
        csrc/k3_attn_f32.cu, K6 LayerNorm) — the arithmetic of the reference without AMP."""
        a = self.self_attention
        wq = torch.cat([a.linear_q.weight, a.linear_k.weight, a.linear_v.weight], 0)
        bq = torch.cat([a.linear_q.bias, a.linear_k.bias, a.linear_v.bias], 0)
        y = ops.BiasedAttentionF32.apply(F.linear(x, wq, bq), bias_slot, layer,
                                         a.attention_dropout_rate if self.training else 0.0, a.scale)    # :1693-1706
        x = x + self.self_attention_dropout(a.output_layer(y))                                           # :1708, :1731-1735
        x = x + self.ffn_dropout(self.ffn(ops.layer_norm(x, self.ffn_norm1)))                            # :1737-1740
        return ops.layer_norm(x, self.ffn_norm2)                                                         # :1741


def gradient_tail_loss(inputs, targets, alpha=0.25, beta=1, k=1):
    """model_fqandtoyo.py:545-550 — the K7 kernel (csrc/k7_loss.cu); only the reference's own beta = k = 1 is built."""
    if beta != 1 or k != 1:
        raise NotImplementedError("GradientTailLoss: libmobgt implements beta = 1, k = 1 (the only values the reference uses)")
    return ops.gradient_tail_loss(inputs, targets, alpha)


class Graphormer(nn.Module):
    def __init__(self, n_layers, num_heads, hidden_dim, dropout_rate, intput_dropout_rate, weight_decay, ffn_dim,
                 dataset_name, warmup_updates, tot_updates, peak_lr, end_lr, edge_type, multi_hop_max_dist,
                 attention_dropout_rate, flag=False, flag_m=3, flag_step_size=1e-3, flag_mag=1e-3, lr_step=2, world=None,
                 tf32=True, precision=16):
        """precision: the pl.Trainer flag of the reference (README.md:62 runs `--precision 16`).  16: bf16 GEMMs / attention on
        the tensor cores, fp32 residual stream, LayerNorms and losses (the AMP split; parity 2e-2).  32: fp32 operands and
        arithmetic everywhere — IEEE fp32 GEMMs, fp32 attention kernels (csrc/k3_attn_f32.cu), fp32 bias; parity 1e-5 against
        the reference's fp32 statement.  It is the full-precision / verification mode, not the benchmarked one.
        tf32: run the GEMMs that stay in fp32 storage (GCN dense parts modelGNN.py:39, user fuse, cat_decoder, out_proj) on
        the TF32 tensor cores instead of SIMT FFMA.  The reference runs them in fp16 under `--precision 16` autocast
        (README.md:62), so TF32 (10-bit mantissa, fp32 range and accumulate) is at least as precise; tf32=False keeps IEEE fp32."""
        super().__init__()
        if precision not in (16, 32):
            raise NotImplementedError(f"precision={precision!r}: 16 (bf16 tensor-core path) or 32 (fp32 path)")
        self.precision = int(precision)
        self.tf32 = bool(tf32) and self.precision == 16
        ops.enable_tf32(self.tf32)          # precision=32 asks for IEEE fp32 GEMMs (forward AND backward: a process-wide switch)
        if world is None:
            raise ValueError("Graphormer needs a PoiWorld (the dataset tables the reference reads from ../dataset/<name>/raw, "
                             "model_fqandtoyo.py:791-832)")
        if dataset_name not in DATASET_TRAITS:
            raise NotImplementedError(f"dataset_name={dataset_name!r}: only the POI graph datasets are on the MobGT hot path")
        if (num_heads, hidden_dim) not in SUPPORTED_SHAPES or (hidden_dim + 64) % num_heads:
            raise NotImplementedError(
                f"num_heads={num_heads}, hidden_dim={hidden_dim}: libmobgt is built for (num_heads, hidden_dim) in "
                f"{sorted(SUPPORTED_SHAPES)}. The encoder width is hidden_dim + 64 (time and category embeddings), split over the "
                f"heads: the attention-bias kernels (K2) are built for 8 heads and for 12 heads, and the attention kernels (K3) "
                f"for head dims {ops.HEAD_DIMS[0]} and {ops.HEAD_DIMS[1]}, i.e. hidden_dim 64 or 128 at 8 heads and hidden_dim "
                f"128 at 12 heads.")
        tr = DATASET_TRAITS[dataset_name]
        self.traits, self.dataset_name = tr, dataset_name
        self.num_virtual_tokens, self.num_heads, self.hidden_dim = 1, num_heads, hidden_dim
        self.time_embed_dim = self.cat_embed_dim = 32
        H, C, P = num_heads, world.C, world.P
        D = hidden_dim + self.time_embed_dim + self.cat_embed_dim
        # edge_type "multi_hop" (README.md:62): the mean over the shortest path of edge_encoder rows through edge_dis_encoder;
        # any other value: Graphormer's direct encoding, edge_encoder[attn_edge_type] (edge_dis_encoder is kept, unused, so
        # that both modes have the same state_dict)
        self.edge_type, self.multi_hop_max_dist = edge_type, multi_hop_max_dist
        self.direct_edges = edge_type != "multi_hop"
        self.edge_encoder = nn.Embedding(128, H, padding_idx=0)
        self.edge_dis_encoder = nn.Embedding(128 * H * H, 1)
        self.rel_pos_encoder = nn.Embedding(512, H, padding_idx=0)
        self.poi_distance_model = GCN(3 + C, [16, 64], hidden_dim, 0.3)
        self.poi_cat_model = GCN(C, [16, 64], self.cat_embed_dim, 0.1)
        self.user_embed_model = UserEmbeddings(world.U + tr["user_extra"], hidden_dim)
        self.time_embed_model_48 = nn.Embedding(tr["time_rows"], self.time_embed_dim, padding_idx=tr["time_pad"])
        self.cat_decoder = nn.Linear(2 * hidden_dim + 64, C + tr["cat_extra"])
        self.embed_fuse_model2 = FuseEmbeddings(hidden_dim, self.time_embed_dim)
        self.embed_fuse_model3 = FuseEmbeddings(hidden_dim, D)
        self.embed_fuse_model4 = FuseEmbeddings(hidden_dim + self.time_embed_dim, self.cat_embed_dim)
        self.pos_embed = LearnablePositionalEncoding(NODE_DIM, D)
        self.in_degree_encoder = nn.Embedding(128, D, padding_idx=0)
        self.out_degree_encoder = nn.Embedding(128, D, padding_idx=0)
        self.fre_embed_model = nn.Embedding(int(world.check_freq.max()) + 1, D, padding_idx=0)   # only row 0 (== 0) is ever read
        self.poi_pos_encoder = nn.Embedding(world.num_bins, H, padding_idx=0)
        self.input_dropout = nn.Dropout(intput_dropout_rate)
        self.output_dropout = nn.Dropout(intput_dropout_rate)
        self.layers = nn.ModuleList([EncoderLayer(D, ffn_dim, dropout_rate, attention_dropout_rate, H) for _ in range(n_layers)])
        self._w16 = ops.Bf16Weights()          # bf16 working copies of the encoder's Linear parameters
        for li, layer in enumerate(self.layers):
            a = layer.self_attention
            self._w16.register((li, "qkv"), [a.linear_q, a.linear_k, a.linear_v])
            self._w16.register((li, "o"), [a.output_layer])
            self._w16.register((li, "f1"), [layer.ffn.layer1])
            self._w16.register((li, "f2"), [layer.ffn.layer2])
        self._w16.register(("emb", "fuse2"), [self.embed_fuse_model2.fuse_embed])
        self._w16.register(("emb", "fuse4"), [self.embed_fuse_model4.fuse_embed])
        self.final_ln = nn.LayerNorm(2 * hidden_dim + 64)
        self.out_proj = nn.Linear(2 * hidden_dim + 64, P + tr["poi_extra"])
        self._w16.register(("head", "out"), [self.out_proj], pad_rows_to=8)   # training head: bf16 GEMM (fp16 under the reference's AMP)
        self.ELU = nn.ELU()
        self.graph_token = nn.Embedding(1, D)
        self.graph_token_virtual_distance = nn.Embedding(1, H)
        self.warmup_updates, self.tot_updates, self.peak_lr, self.end_lr = warmup_updates, tot_updates, peak_lr, end_lr
        self.weight_decay, self.lr_step = weight_decay, lr_step
        self.flag, self.flag_m, self.flag_step_size, self.flag_mag = flag, flag_m, flag_step_size, flag_mag
        self.metric, self.cat_target = "NLLLoss", None
        # dataset tables (non-trainable)
        self.register_buffer("X", torch.from_numpy(world.X), persistent=False)
        self.register_buffer("C_X", torch.from_numpy(world.C_X), persistent=False)
        self._x_sparse = {}
        for name, dense in (("X", world.X), ("C_X", world.C_X)):     # constant, mostly-zero input features -> CSR for K8
            d = np.asarray(dense, np.float32)
            if (d != 0).mean() <= 0.125:
                csr = _dense_to_csr(d)
                chunked, fold = _csr_split_rows(_csr_transpose(csr, d.shape[0], d.shape[1]))   # X^T has a few very long rows
                for suffix, (crow, col, val) in (("", csr), ("_t", chunked), ("_f", fold)):
                    self.register_buffer(f"{name}s{suffix}_crow", torch.from_numpy(np.ascontiguousarray(crow, np.int32)), persistent=False)
                    self.register_buffer(f"{name}s{suffix}_col", torch.from_numpy(np.ascontiguousarray(col, np.int32)), persistent=False)
                    self.register_buffer(f"{name}s{suffix}_val", torch.from_numpy(np.ascontiguousarray(val, np.float32)), persistent=False)
                self._x_sparse[name] = True
        self.register_buffer("cat_of_poi", torch.from_numpy(world.cat_of_poi).int(), persistent=False)
        for name, csr, n in (("D_A", world.D_A, P), ("C_A", world.C_A, C)):
            for suffix, (crow, col, val) in (("", csr), ("_t", _csr_transpose(csr, n))):
                self.register_buffer(f"{name}{suffix}_crow", torch.from_numpy(np.ascontiguousarray(crow, np.int32)), persistent=False)
                self.register_buffer(f"{name}{suffix}_col", torch.from_numpy(np.ascontiguousarray(col, np.int32)), persistent=False)
                self.register_buffer(f"{name}{suffix}_val", torch.from_numpy(np.ascontiguousarray(val, np.float32)), persistent=False)

    # ------------------------------------------------------------------------------------------
    def _adj(self, name):
        """(A, A^T) as CSR triples (crow i32, col i32, val f32) — the operands of K8."""
        t = lambda s: (getattr(self, f"{name}{s}_crow"), getattr(self, f"{name}{s}_col"), getattr(self, f"{name}{s}_val"))
        return t(""), t("_t")

    def gcn_tables(self):
        """model_fqandtoyo.py:1236-1237: recomputed every forward, like the reference."""
        t = lambda n, sfx: tuple(getattr(self, f"{n}s{sfx}_{k}") for k in ("crow", "col", "val"))
        xs = lambda n: (t(n, ""), (t(n, "_t"), t(n, "_f"))) if self._x_sparse.get(n) else None
        return (self.poi_distance_model(self.X, self._adj("D_A"), xs("X")), self.poi_cat_model(self.C_X, self._adj("C_A"), xs("C_X")))

    def attn_bias(self, b, dtype=torch.bfloat16):
        """K2 (model_fqandtoyo.py:1143-1216)"""
        return ops.AttnBias.apply(b, self.rel_pos_encoder.weight, self.poi_pos_encoder.weight, self.edge_encoder.weight,
                                  self.edge_dis_encoder.weight, self.graph_token_virtual_distance.weight, dtype, self.direct_edges)

    def node_tokens(self, b, dtype=torch.bfloat16):
        """K4 (model_fqandtoyo.py:1222-1344) -> packed tokens [ntok, hidden_dim + 64]"""
        Gd, Gc = self.gcn_tables()
        e = ops.EmbedGather.apply(b, self.cat_of_poi, Gd, self.time_embed_model_48.weight, Gc, dtype, self.traits["time_pad"])
        hp = self.hidden_dim + self.time_embed_dim
        f2, f4 = self.embed_fuse_model2.fuse_embed, self.embed_fuse_model4.fuse_embed
        if dtype == torch.bfloat16:     # bf16 working copies of the weights, bias gradients through the K6 column sum
            self._w16.refresh()
            x = F.leaky_relu(ops.linear_bf16(e[:, :hp], f2, *self._w16.get(("emb", "fuse2"))), 0.2)      # :1268
            x = F.leaky_relu(ops.linear_bf16(torch.cat([x, e[:, hp:]], 1), f4, *self._w16.get(("emb", "fuse4"))), 0.2)   # :1269
        else:
            x = F.leaky_relu(F.linear(e[:, :hp], f2.weight.to(dtype), f2.bias.to(dtype)), 0.2)          # :1268
            x = F.leaky_relu(F.linear(torch.cat([x, e[:, hp:]], 1), f4.weight.to(dtype), f4.bias.to(dtype)), 0.2)   # :1269
        tok = ops.EmbedSum.apply(b, x, self.in_degree_encoder.weight, self.out_degree_encoder.weight, self.pos_embed.pe,
                                 self.graph_token.weight)
        return F.dropout(tok, self.pos_embed.p, self.training)                                           # :358

    def _packed(self, batched_data):
        """The packed Batch1 the kernels consume; a reference-collated dense batch (collator.py:149-215) is converted."""
        if hasattr(batched_data, "rel_pos16"):
            return batched_data
        from .collator import Batch1
        return Batch1.from_dense(batched_data, multi_hop_max_dist=self.multi_hop_max_dist, device=self.X.device)

    def features(self, batched_data):
        """model_fqandtoyo.py:1143-1364 up to the input of the two heads: z [B, 2*hidden+64] fp32 (user fuse of token 0,
        final LayerNorm, ELU, output dropout) — the operand of `out_proj` / `cat_decoder` and of the fused K5 head."""
        b = self._packed(batched_data)
        f32 = self.precision == 32
        tok = self.node_tokens(b, torch.float32 if f32 else torch.bfloat16)
        slot = ops.BiasSlot(b, len(self.layers), dtype=torch.float32 if f32 else torch.bfloat16)
        x = ops.BiasLink.apply(self.input_dropout(tok).float(), slot, self.rel_pos_encoder.weight, self.poi_pos_encoder.weight,
                               self.edge_encoder.weight, self.edge_dis_encoder.weight,
                               self.graph_token_virtual_distance.weight, self.direct_edges)              # K2 (:1143-1216), :1347
        if f32:
            for li, layer in enumerate(self.layers):                                                     # :1348-1352
                x = layer.forward_f32(x, slot, li)
        else:
            x16 = x.to(torch.bfloat16)
            self._w16.refresh()
            for li, layer in enumerate(self.layers):                                                     # :1348-1352
                x, x16 = layer(x, x16, slot, li, self._w16)
        z0 = x.index_select(0, b.tok_off[:-1].long()).float()                                            # output[:, 0, :]
        user_embedding = self.user_embed_model(b.user.view(-1) - 1)                                      # :1239
        z = self.embed_fuse_model3(z0, user_embedding)                                                   # :1356 (token 0 only)
        z = self.output_dropout(self.ELU(ops.layer_norm(z.float(), self.final_ln)))                      # :1360-1364
        self.cat_target = self.cat_of_poi[b.y - 1].long() - 1                                            # :1265
        return z, b

    def forward(self, batched_data, perturb=None):
        z, b = self.features(batched_data)
        cat_output = self.cat_decoder(z)
        output = self.out_proj(z)
        if self.traits["log_softmax"]:
            output = F.log_softmax(output, dim=1)                                                        # :1425
        return [output, cat_output]

    # ------------------------------------------------------------------------------------------ steps
    def training_step(self, batched_data, batch_idx=0, split=False):
        """model_fqandtoyo.py:1434-1478.  The losses are the K7 kernels (csrc/k7_loss.cu): one pass over the logits gives the
        loss, and the same pass of the backward gives d(logits).
        split=True -> (loss, z, z_cut): the autograd graph is cut at z, the [B, 2*hidden+64] input of the two heads.
        `loss.backward()` then runs the head backward only (it completes the gradient of out_proj — 77 of the 92 MB of a c2 model —
        and leaves d loss / d z in z_cut.grad), `z.backward(z_cut.grad)` the encoder backward: the data-parallel trainer captures
        the two halves as two CUDA graphs and all-reduces the out_proj bucket while the second one runs."""
        z, b = self.features(batched_data)
        z_full = z
        if split:
            z = z.detach().requires_grad_(True)
        loss = self._heads_loss(z, b)
        return (loss, z_full, z) if split else loss

    def _heads_loss(self, z, b):
        cat_logits = self.cat_decoder(z)
        # POI logits in bf16 (the reference's `--precision 16` runs this Linear in fp16): [B, P] x 2 bytes instead of 4 through
        # the loss kernels, and a bf16 tensor-core GEMM forward and backward
        # (class count padded to a multiple of 8 with zero weight rows; the loss kernels ignore the padding columns)
        V = self.out_proj.weight.shape[0]
        if self.precision == 32:
            poi_logits = self.out_proj(z)                                                                # fp32 logits through K7
        else:
            poi_logits = ops.linear_bf16(z.to(torch.bfloat16), self.out_proj, *self._w16.get(("head", "out")))
        if self.dataset_name == "toyotagraph":
            loss1 = ops.gradient_tail_loss(cat_logits, self.cat_target, 0.1)                            # :1464-1469
            loss2 = ops.log_softmax_nll_loss(poi_logits, b.y, ignore_index=0, n_classes=V)   # :1425 + data.py:165 NLLLoss(ignore_index=0)
            return loss1 + loss2
        return ops.gradient_tail_loss(poi_logits, b.y - 1, 0.2, n_classes=V)                            # :1447-1460

    def eval_targets(self, batched_data):
        """y_true of validation_step / test_step (model_fqandtoyo.py:1485-1493, 1531-1539): `y - 1` for the datasets in the
        reference's list, plain `y` for toyotagraph (its out_proj has P+1 classes and it trains on y, :1471)."""
        y = batched_data.y
        return y if self.dataset_name == "toyotagraph" else y - 1

    def head_topk(self, z, y_true, k=20, vocab_parallel=None):
        """K5: POI logits + per-row top-k + rank of the target, fused (the logits never reach HBM).  -> dict(idx [B,k] i32,
        val [B,k], rank [B] i32).  log_softmax (toyotagraph, :1425) is monotone per row, so indices and ranks are those of
        the reference's y_pred[0].  vocab_parallel: a process group -> out_proj rows sharded across its ranks, z rows of all
        ranks gathered (SURVEY.md §8e); returns the rows of THIS rank.
        precision 32 ranks IEEE fp32 logits (the fp32 K5 head: fp32 z and the out_proj.weight master itself, no rounding);
        precision 16 ranks bf16-operand logits on the tensor cores."""
        bias = self.out_proj.bias.detach().float()
        t32 = y_true.to(torch.int32).contiguous()
        if self.precision == 32:
            W = self.out_proj.weight.detach()
            zh = z.detach().float().contiguous()
        else:
            W = self.out_proj.weight.detach().to(torch.bfloat16)
            zh = z.detach().to(torch.bfloat16).contiguous()
        if vocab_parallel is None:
            r = ops.head_topk_local(zh, W.contiguous(), bias.contiguous(), t32, k)
            return dict(idx=r["idx"], val=r["val"], rank=r["cnt"])
        from . import parallel
        return parallel.vocab_parallel_eval_head(ops, zh, W, bias, t32, k, vocab_parallel)

    def _eval_step(self, batched_data, full_logits, vocab_parallel):
        z, b = self.features(batched_data)
        y_true = self.eval_targets(b)
        out = {"y_true": y_true, "idx": b.idx}
        out.update(self.head_topk(z, y_true, 20, vocab_parallel))
        if full_logits:                    # the reference's return value (a [B, P] tensor per batch); off on the fast path
            output = self.out_proj(z)
            out["y_pred"] = [F.log_softmax(output, dim=1) if self.traits["log_softmax"] else output, self.cat_decoder(z)]
        return out

    def validation_step(self, batched_data, batch_idx=0, full_logits=False, vocab_parallel=None):
        """model_fqandtoyo.py:1484-1496, through the fused head: returns y_true plus top-20 indices and the target's rank."""
        out = self._eval_step(batched_data, full_logits, vocab_parallel)
        out.pop("idx")
        return out

    def test_step(self, batched_data, batch_idx=0, full_logits=False, vocab_parallel=None):
        """model_fqandtoyo.py:1530-1544"""
        return self._eval_step(batched_data, full_logits, vocab_parallel)

    def test_epoch_end(self, outputs, group=None, quiet=False):
        """model_fqandtoyo.py:1546-1597: Acc@{1,5,10,20}, NDCG@k, MRR over all batches (of all ranks: the per-batch SUMS are
        all-reduced, the reference's `sync_dist=True`); prints the reference's three lines on rank 0."""
        from . import parallel
        tot, n = {}, 0
        for o in outputs:
            m = ops.metrics_from_rank(o["rank"], o["y_true"])      # per batch: keeps get_acc's break at the first target == 0
            for k_, v in m.items():
                tot[k_] = tot.get(k_, 0.0) + v
            n += len(o["y_true"])
        if not tot:
            tot = {f"{a}{k_}": 0.0 for a in ("acc", "ndcg") for k_ in (1, 5, 10, 20)}
            tot["mrr"] = 0.0
        tot, n = parallel.reduce_metric_sums(tot, n, group=group, device=self.X.device)
        avg = {k_: v / max(n, 1) for k_, v in tot.items()}
        if not quiet and parallel.is_rank0(group):
            print(f"ACC @1: {round(avg['acc1'], 4)}, @5: {round(avg['acc5'], 4)}, @10: {round(avg['acc10'], 4)}")
            print(f"NDCG @1: {round(avg['ndcg1'], 4)}, @5: {round(avg['ndcg5'], 4)}, @10: {round(avg['ndcg10'], 4)}")
            print(f"MRR: {round(avg['mrr'], 4)}")
        avg["n"] = n
        return avg

    validation_epoch_end = test_epoch_end

    def _flat_param_order(self):
        """All parameters, with the q / k / v weights (and biases) of every attention layer next to each other: their gradients
        then lie back to back in the flat gradient buffer, and the fused QKV backward writes dW [3 x hidden, hidden] and db with
        ONE GEMM / column-sum output (ops._claim)."""
        fused, seen = [], set()
        for layer in self.layers:
            a = layer.self_attention
            fused += [a.linear_q.weight, a.linear_k.weight, a.linear_v.weight, a.linear_q.bias, a.linear_k.bias, a.linear_v.bias]
        seen = {id(p) for p in fused} | {id(self.out_proj.weight)}
        # out_proj.weight LAST: its gradient (77 of 92 MB at P = 60 000) is all-reduced on its own, early (trainer.Trainer); with
        # the bucket at the end of the flat buffer the remainder is ONE contiguous all-reduce instead of two
        return fused + [p for p in self.parameters() if id(p) not in seen] + [self.out_proj.weight]

    def configure_optimizers(self):
        """model_fqandtoyo.py:1599-1616"""
        params = self._flat_param_order()
        if params[0].is_cuda:        # K9: one kernel over flat parameter / gradient buffers (same arithmetic as torch's AdamW)
            from .optim import FlatAdamW
            optimizer = FlatAdamW(params, lr=self.peak_lr, weight_decay=self.weight_decay)
        else:
            optimizer = torch.optim.AdamW(params, lr=self.peak_lr, weight_decay=self.weight_decay)
        sched = PolynomialDecayLR(optimizer, warmup_updates=self.warmup_updates, tot_updates=self.tot_updates, lr=self.peak_lr,
                                  end_lr=self.end_lr, power=1.0)
        return [optimizer], [{"scheduler": sched, "name": "learning_rate", "interval": "step", "frequency": 1}]

    @staticmethod
    def add_model_specific_args(parent_parser):
        """model_fqandtoyo.py:1618-1641 (same names, defaults and the reference's own typo)."""
        parser = parent_parser.add_argument_group("Graphormer")
        parser.add_argument("--n_layers", type=int, default=12)
        parser.add_argument("--num_heads", type=int, default=32)
        parser.add_argument("--hidden_dim", type=int, default=512)
        parser.add_argument("--ffn_dim", type=int, default=512)
        parser.add_argument("--intput_dropout_rate", type=float, default=0.1)
        parser.add_argument("--dropout_rate", type=float, default=0.1)
        parser.add_argument("--weight_decay", type=float, default=0.01)
        parser.add_argument("--attention_dropout_rate", type=float, default=0.1)
        parser.add_argument("--checkpoint_path", type=str, default="")
        parser.add_argument("--warmup_updates", type=int, default=60000)
        parser.add_argument("--tot_updates", type=int, default=1000000)
        parser.add_argument("--peak_lr", type=float, default=2e-4)
        parser.add_argument("--end_lr", type=float, default=1e-9)
        parser.add_argument("--edge_type", type=str, default="multi_hop")
        parser.add_argument("--validate", action="store_true", default=False)
        parser.add_argument("--test", action="store_true", default=False)
        parser.add_argument("--flag", action="store_true")
        parser.add_argument("--flag_m", type=int, default=3)
        parser.add_argument("--flag_step_size", type=float, default=1e-3)
        parser.add_argument("--flag_mag", type=float, default=1e-3)
        return parent_parser
