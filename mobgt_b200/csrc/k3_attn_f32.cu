// K3 (fp32 mode) — the biased attention of model_fqandtoyo.py:1693-1706 and its backward with fp32 operands, fp32 bias and
// fp32 results, for graphs of any size up to 1 025 tokens.
//
// Why: the contract of this path is "within 1e-5 relative in fp32 mode, 2e-2 in bf16 mode" against the reference's own
// arithmetic.  The tensor-core kernels (k3_attn_fwd.cu / k3_attn_bwd.cu) round Q, K, V, the bias and the probabilities to bf16
// by construction, so they can only carry the second half of that sentence.  These kernels are the first half: the model's
// `precision=32` mode (the reference's Lightning default, `--precision 32`) runs its attention here, and the parity tests
// compare logits, loss and every parameter gradient with the fp32 oracle at 1e-5.  It is a verification / full-precision
// mode, not the benchmarked one: plain SIMT FFMA, one CTA per (graph, head), IEEE expf / logf.
//
// Layout: K and V (backward: Q, K, V, dO) of the (graph, head) are staged in shared memory with an odd row pitch of d + 1 floats
// (25 for head dim 24, 17 for 16: lanes read different rows, conflict-free); a warp owns one query row (forward and the dQ / dS
// pass) or one key column (the dK / dV pass) at a time, its lanes stride over the other index, and the d-wide partial sums are
// merged by shuffles in a fixed
// order — no atomics, bitwise reproducible.  The backward stages Q, K, V and dO together (4 T (d + 1) floats), which fits up to
// T = 513; a batch with a larger graph runs the backward as two kernels that stage half each (k3_attn_large.cu, float
// instantiation: the same expressions in the same order, so the same bits).  Scores and probabilities are recomputed, never stored.  The dropout mask is the
// tensor-core path's (common.cuh attn_drop_*: same seed, same mask).
#include "common.cuh"
#include "k3_small.cuh"

namespace mobgt {

namespace {
constexpr int kWarps = 8;
constexpr int kThreadsF = kWarps * 32;
constexpr int kMaxT = MOBGT_MAX_MODEL_NODES + 1;   // forward: 2 T (d + 1) floats of shared memory, 205 KB at T = 1025

struct F32AttnParams {
    const int32_t *tok_off;
    const float *q, *k, *v;       // [ntok, qkv_stride]
    int64_t qkv_stride;
    const float *bias;            // [B,H,T,Tp]
    int H, T, Tp;
    float scale;
    AttnDrop drop;
    float *out, *lse;             // [ntok, H*d], [ntok, H]  (backward: o / lse are inputs)
    const float *o, *dout;
    float *dq, *dk, *dv;
    int64_t dqkv_stride;
    float *dbias;                 // f32 [B,H,T,Tp]
    int accumulate;               // 0: overwritten, 1: added to
};

__device__ __forceinline__ float warp_sum(float x) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xFFFFFFFFu, x, o);
    return x;
}
__device__ __forceinline__ float warp_max(float x) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) x = fmaxf(x, __shfl_xor_sync(0xFFFFFFFFu, x, o));
    return x;
}
// rows [t0, t0 + Tg) x d floats of head h of a [ntok, stride] matrix -> dst[row * (d + 1) + e]
template <int kD, int kPitch = kD + 1>
__device__ __forceinline__ void stage(const float *src, int64_t stride, int t0, int Tg, int h, float *dst) {
    for (int i = threadIdx.x; i < Tg * kD; i += kThreadsF) {
        const int r = i / kD, e = i - r * kD;
        dst[r * kPitch + e] = __ldg(src + (size_t)(t0 + r) * stride + h * kD + e);
    }
}
template <int kD>
__device__ __forceinline__ float dotd(const float (&a)[kD], const float *b) {
    float s = 0.f;
#pragma unroll
    for (int e = 0; e < kD; ++e) s = fmaf(a[e], b[e], s);
    return s;
}
__device__ __forceinline__ bool keep_bit(bool on, uint32_t rowkey, int col, uint32_t th16) {
    return !on || ((attn_drop_keep8(rowkey, (uint32_t)(col >> 3), th16) >> (col & 7)) & 1u);
}

}  // namespace

// ---------------------------------------------------------------------------------------------------------------- forward
template <int kD>
__global__ void __launch_bounds__(kThreadsF) k3f_attn_fwd_kernel(const F32AttnParams p) {
    constexpr int kPitch = kD + 1;
    extern __shared__ __align__(16) float smem[];
    const int g = blockIdx.x / p.H, h = blockIdx.x - g * p.H;
    const int t0 = p.tok_off[g], Tg = p.tok_off[g + 1] - t0;
    if (Tg <= 0) return;
    float *sK = smem, *sV = smem + Tg * kPitch;
    stage<kD>(p.k, p.qkv_stride, t0, Tg, h, sK);
    stage<kD>(p.v, p.qkv_stride, t0, Tg, h, sV);
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const bool drop = p.drop.th16 != 0;
    uint32_t seed_lo = 0, seed_hi = 0;
    if (drop) attn_drop_fold_seed(p.drop, seed_lo, seed_hi);
    const int plane = g * p.H + h;
    for (int i = warp; i < Tg; i += kWarps) {
        float q[kD];
        const float *qg = p.q + (size_t)(t0 + i) * p.qkv_stride + h * kD;
#pragma unroll
        for (int e = 0; e < kD; ++e) q[e] = __ldg(qg + e);
        const float *brow = p.bias + ((size_t)plane * p.T + i) * p.Tp;
        const uint32_t rowkey = drop ? attn_drop_rowkey((uint32_t)plane, (uint32_t)i, seed_lo, seed_hi) : 0u;
        float m = -INFINITY;
        for (int j = lane; j < Tg; j += 32) m = fmaxf(m, fmaf(p.scale, dotd(q, sK + j * kPitch), __ldg(brow + j)));
        m = warp_max(m);
        float l = 0.f, o[kD];
#pragma unroll
        for (int e = 0; e < kD; ++e) o[e] = 0.f;
        for (int j = lane; j < Tg; j += 32) {
            const float pe = expf(fmaf(p.scale, dotd(q, sK + j * kPitch), __ldg(brow + j)) - m);
            l += pe;                                          // the denominator is taken before the dropout mask
            if (keep_bit(drop, rowkey, j, p.drop.th16)) {
                const float *vr = sV + j * kPitch;
#pragma unroll
                for (int e = 0; e < kD; ++e) o[e] = fmaf(pe, vr[e], o[e]);
            }
        }
        l = warp_sum(l);
        const float inv = (drop ? p.drop.inv_keep : 1.0f) / l;
        float mine = 0.f;
#pragma unroll
        for (int e = 0; e < kD; ++e) {
            const float s = warp_sum(o[e]);
            if (lane == e) mine = s;
        }
        if (lane < kD) p.out[(size_t)(t0 + i) * (p.H * kD) + h * kD + lane] = mine * inv;
        if (lane == 0) p.lse[(size_t)(t0 + i) * p.H + h] = m + logf(l);
    }
}

// ---------------------------------------------------------------------------------------------------------------- backward
// pass A, warp = query row i: D_i = dO_i . O_i ; per key j: p = exp(s - lse_i), dP = dO_i . V_j (masked, / keep),
//         dS = p (dP - D_i) -> dbias, dQ_i = scale * sum_j dS K_j
// pass B, warp = key column j: the same p / dS recomputed per query row i: dK_j = scale * sum_i dS Q_i, dV_j = sum_i (mask p / keep) dO_i
template <int kD>
__global__ void __launch_bounds__(kThreadsF) k3f_attn_bwd_kernel(const F32AttnParams p) {
    constexpr int kPitch = kD + 1;
    extern __shared__ __align__(16) float smem[];
    const int g = blockIdx.x / p.H, h = blockIdx.x - g * p.H;
    const int t0 = p.tok_off[g], Tg = p.tok_off[g + 1] - t0;
    if (Tg <= 0) return;
    const int HD = p.H * kD;
    float *sQ = smem, *sK = sQ + Tg * kPitch, *sV = sK + Tg * kPitch, *sdO = sV + Tg * kPitch;
    float *sLse = sdO + Tg * kPitch, *sDel = sLse + Tg;
    stage<kD>(p.q, p.qkv_stride, t0, Tg, h, sQ);
    stage<kD>(p.k, p.qkv_stride, t0, Tg, h, sK);
    stage<kD>(p.v, p.qkv_stride, t0, Tg, h, sV);
    stage<kD>(p.dout, HD, t0, Tg, h, sdO);
    for (int i = threadIdx.x; i < Tg; i += kThreadsF) {
        const float *og = p.o + (size_t)(t0 + i) * HD + h * kD, *dg = p.dout + (size_t)(t0 + i) * HD + h * kD;
        float d = 0.f;
#pragma unroll
        for (int e = 0; e < kD; ++e) d = fmaf(__ldg(og + e), __ldg(dg + e), d);
        sDel[i] = d;
        sLse[i] = p.lse[(size_t)(t0 + i) * p.H + h];
    }
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const bool drop = p.drop.th16 != 0;
    const float ik = drop ? p.drop.inv_keep : 1.0f;
    uint32_t seed_lo = 0, seed_hi = 0;
    if (drop) attn_drop_fold_seed(p.drop, seed_lo, seed_hi);
    const int plane = g * p.H + h;
    const size_t pl = (size_t)plane * p.T * p.Tp;
    // ---- pass A
    for (int i = warp; i < Tg; i += kWarps) {
        float q[kD], dO[kD], dq[kD];
#pragma unroll
        for (int e = 0; e < kD; ++e) {
            q[e] = sQ[i * kPitch + e];
            dO[e] = sdO[i * kPitch + e];
            dq[e] = 0.f;
        }
        const float lse = sLse[i], del = sDel[i];
        const uint32_t rowkey = drop ? attn_drop_rowkey((uint32_t)plane, (uint32_t)i, seed_lo, seed_hi) : 0u;
        const float *brow = p.bias + pl + (size_t)i * p.Tp;
        float *drow = p.dbias + pl + (size_t)i * p.Tp;
        for (int j = lane; j < Tg; j += 32) {
            const float *kr = sK + j * kPitch;
            const float pr = expf(fmaf(p.scale, dotd(q, kr), __ldg(brow + j)) - lse);
            const float dp = keep_bit(drop, rowkey, j, p.drop.th16) ? dotd(dO, sV + j * kPitch) * ik : 0.f;
            const float ds = pr * (dp - del);
            drow[j] = (p.accumulate == 1 ? drow[j] : 0.f) + ds;
#pragma unroll
            for (int e = 0; e < kD; ++e) dq[e] = fmaf(ds, kr[e], dq[e]);
        }
        float mine = 0.f;
#pragma unroll
        for (int e = 0; e < kD; ++e) {
            const float s = warp_sum(dq[e]);
            if (lane == e) mine = s;
        }
        if (lane < kD) p.dq[(size_t)(t0 + i) * p.dqkv_stride + h * kD + lane] = mine * p.scale;
    }
    // ---- pass B
    for (int j = warp; j < Tg; j += kWarps) {
        float k[kD], v[kD], dk[kD], dv[kD];
#pragma unroll
        for (int e = 0; e < kD; ++e) {
            k[e] = sK[j * kPitch + e];
            v[e] = sV[j * kPitch + e];
            dk[e] = dv[e] = 0.f;
        }
        for (int i = lane; i < Tg; i += 32) {
            const float *qr = sQ + i * kPitch, *dor = sdO + i * kPitch;
            const float pr = expf(fmaf(p.scale, dotd(k, qr), __ldg(p.bias + pl + (size_t)i * p.Tp + j)) - sLse[i]);
            bool kp = true;
            if (drop) kp = keep_bit(true, attn_drop_rowkey((uint32_t)plane, (uint32_t)i, seed_lo, seed_hi), j, p.drop.th16);
            const float pd = kp ? pr * ik : 0.f;
            const float ds = pr * ((kp ? dotd(v, dor) * ik : 0.f) - sDel[i]);
#pragma unroll
            for (int e = 0; e < kD; ++e) {
                dk[e] = fmaf(ds, qr[e], dk[e]);
                dv[e] = fmaf(pd, dor[e], dv[e]);
            }
        }
        float mk = 0.f, mv = 0.f;
#pragma unroll
        for (int e = 0; e < kD; ++e) {
            const float a = warp_sum(dk[e]), b = warp_sum(dv[e]);
            if (lane == e) { mk = a; mv = b; }
        }
        if (lane < kD) {
            p.dk[(size_t)(t0 + j) * p.dqkv_stride + h * kD + lane] = mk * p.scale;
            p.dv[(size_t)(t0 + j) * p.dqkv_stride + h * kD + lane] = mv;
        }
    }
}

namespace {
int32_t check_common(const void *q, const void *k, const void *v, const void *bias, const int32_t *tok_off, int32_t B, int32_t H,
                     int32_t ntok, int32_t T, int32_t Tp, int32_t t_max_host, float drop_p) {
    MOBGT_REQUIRE(q && k && v && bias && tok_off, MOBGT_ERR_NULL, "mobgt_attn_f32: null pointer");
    MOBGT_REQUIRE(B >= 0 && H > 0 && ntok >= 0 && T > 0 && Tp >= T, MOBGT_ERR_BAD_SHAPE, "mobgt_attn_f32: bad sizes B=%d H=%d ntok=%d T=%d Tp=%d", B,
                  H, ntok, T, Tp);
    MOBGT_REQUIRE(t_max_host >= 1 && t_max_host <= T && T <= kMaxT, MOBGT_ERR_BAD_SHAPE,
                  "mobgt_attn_f32: t_max_host=%d must be in [1, T=%d] and T <= %d (graphs of at most 1024 nodes)", t_max_host, T, kMaxT);
    MOBGT_REQUIRE(drop_p >= 0.f && drop_p < 1.f, MOBGT_ERR_BAD_SHAPE, "mobgt_attn_f32: drop_p=%f outside [0, 1)", (double)drop_p);
    return MOBGT_OK;
}
}  // namespace

}  // namespace mobgt

using namespace mobgt;

extern "C" int32_t mobgt_attn_f32_fwd_hd(const float *q, const float *k, const float *v, int64_t qkv_row_stride, const float *bias,
                                         const int32_t *tok_off, int32_t B, int32_t H, int32_t ntok, int32_t T, int32_t Tp,
                                         int32_t t_max_host, float scale, float drop_p, uint64_t seed, const void *seed_dev, float *out,
                                         float *lse, int32_t head_dim, void *stream) {
    MOBGT_REQUIRE(head_dim == 16 || head_dim == 24, MOBGT_ERR_UNSUPPORTED,
                  "mobgt_attn_f32_fwd_hd: head_dim=%d is not built (head dims 16 and 24)", head_dim);
    const int32_t rc = check_common(q, k, v, bias, tok_off, B, H, ntok, T, Tp, t_max_host, drop_p);
    if (rc != MOBGT_OK) return rc;
    MOBGT_REQUIRE(out && lse, MOBGT_ERR_NULL, "mobgt_attn_f32_fwd: null output");
    if (B == 0 || ntok == 0) return MOBGT_OK;
    F32AttnParams p{};
    p.tok_off = tok_off; p.q = q; p.k = k; p.v = v; p.qkv_stride = qkv_row_stride; p.bias = bias;
    p.H = H; p.T = T; p.Tp = Tp; p.scale = scale; p.drop = make_attn_drop(drop_p, seed, seed_dev);
    p.out = out; p.lse = lse;
    const size_t smem = (size_t)2 * t_max_host * (head_dim + 1) * sizeof(float);    // row pitch d + 1
    auto kern = head_dim == 16 ? k3f_attn_fwd_kernel<16> : k3f_attn_fwd_kernel<24>;
    MOBGT_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<B * H, kThreadsF, smem, static_cast<cudaStream_t>(stream)>>>(p);
    MOBGT_LAUNCH_OK("k3f_attn_fwd_kernel");
    return MOBGT_OK;
}

extern "C" int32_t mobgt_attn_f32_bwd_hd(const float *q, const float *k, const float *v, int64_t qkv_row_stride, const float *bias,
                                         const float *o, const float *dout, const float *lse, const int32_t *tok_off, int32_t B,
                                         int32_t H, int32_t ntok, int32_t T, int32_t Tp, int32_t t_max_host, float scale, float *dq,
                                         float *dk, float *dv, int64_t dqkv_row_stride, float *dbias, int32_t mode, float drop_p,
                                         uint64_t seed, const void *seed_dev, int32_t head_dim, void *stream) {
    MOBGT_REQUIRE(head_dim == 16 || head_dim == 24, MOBGT_ERR_UNSUPPORTED,
                  "mobgt_attn_f32_bwd_hd: head_dim=%d is not built (head dims 16 and 24)", head_dim);
    const int32_t rc = check_common(q, k, v, bias, tok_off, B, H, ntok, T, Tp, t_max_host, drop_p);
    if (rc != MOBGT_OK) return rc;
    MOBGT_REQUIRE(o && dout && lse && dq && dk && dv && dbias, MOBGT_ERR_NULL, "mobgt_attn_f32_bwd: null pointer");
    MOBGT_REQUIRE(mode == 0 || mode == 1, MOBGT_ERR_BAD_SHAPE, "mobgt_attn_f32_bwd: mode=%d (0: dbias overwritten, 1: added to)", mode);
    if (B == 0 || ntok == 0) return MOBGT_OK;
    F32AttnParams p{};
    p.tok_off = tok_off; p.q = q; p.k = k; p.v = v; p.qkv_stride = qkv_row_stride; p.bias = bias;
    p.H = H; p.T = T; p.Tp = Tp; p.scale = scale; p.drop = make_attn_drop(drop_p, seed, seed_dev);
    p.lse = const_cast<float *>(lse); p.o = o; p.dout = dout; p.dq = dq; p.dk = dk; p.dv = dv; p.dqkv_stride = dqkv_row_stride;
    p.dbias = dbias; p.accumulate = mode;
    if (t_max_host > kLargeT) {
        LargeAttnParams lp{};
        lp.tok_off = tok_off; lp.q = q; lp.k = k; lp.v = v; lp.qkv_stride = qkv_row_stride; lp.bias = bias;
        lp.H = H; lp.T = T; lp.Tp = Tp; lp.scale = scale; lp.t_lo = 0; lp.drop = p.drop;
        lp.lse = p.lse; lp.o = o; lp.dout = dout; lp.dq = dq; lp.dk = dk; lp.dv = dv; lp.dqkv_stride = dqkv_row_stride;
        lp.dbias = dbias; lp.accumulate = mode;
        auto f = head_dim == 16 ? launch_large_attn_bwd<float, 16> : launch_large_attn_bwd<float, 24>;
        return f(lp, B, t_max_host, static_cast<cudaStream_t>(stream));
    }
    const size_t smem = ((size_t)4 * t_max_host * (head_dim + 1) + 2 * (size_t)t_max_host) * sizeof(float);   // row pitch d + 1
    auto kern = head_dim == 16 ? k3f_attn_bwd_kernel<16> : k3f_attn_bwd_kernel<24>;
    MOBGT_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<B * H, kThreadsF, smem, static_cast<cudaStream_t>(stream)>>>(p);
    MOBGT_LAUNCH_OK("k3f_attn_bwd_kernel");
    return MOBGT_OK;
}

extern "C" int32_t mobgt_attn_f32_fwd(const float *q, const float *k, const float *v, int64_t qkv_row_stride, const float *bias,
                                      const int32_t *tok_off, int32_t B, int32_t H, int32_t ntok, int32_t T, int32_t Tp,
                                      int32_t t_max_host, float scale, float drop_p, uint64_t seed, const void *seed_dev, float *out,
                                      float *lse, void *stream) {
    return mobgt_attn_f32_fwd_hd(q, k, v, qkv_row_stride, bias, tok_off, B, H, ntok, T, Tp, t_max_host, scale, drop_p, seed, seed_dev,
                                 out, lse, 24, stream);
}

extern "C" int32_t mobgt_attn_f32_bwd(const float *q, const float *k, const float *v, int64_t qkv_row_stride, const float *bias,
                                      const float *o, const float *dout, const float *lse, const int32_t *tok_off, int32_t B,
                                      int32_t H, int32_t ntok, int32_t T, int32_t Tp, int32_t t_max_host, float scale, float *dq,
                                      float *dk, float *dv, int64_t dqkv_row_stride, float *dbias, int32_t mode, float drop_p,
                                      uint64_t seed, const void *seed_dev, void *stream) {
    return mobgt_attn_f32_bwd_hd(q, k, v, qkv_row_stride, bias, o, dout, lse, tok_off, B, H, ntok, T, Tp, t_max_host, scale, dq, dk,
                                 dv, dqkv_row_stride, dbias, mode, drop_p, seed, seed_dev, 24, stream);
}
