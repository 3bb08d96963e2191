// K3 for graphs of 513 to 1 024 nodes (514 .. 1 025 tokens): the biased attention of model_fqandtoyo.py:1693-1706 and its
// backward, on the CUDA cores.
//
// Why SIMT: such graphs are rare (2 of 4 970 Gowalla-Nevada train trajectories, at most one per 256-graph batch) and the
// tensor-core kernels are sized for T <= 513 (K/V of a graph and every dQ tile resident; two CTAs per SM).  These kernels take
// the large graphs of a batch on the device (Tg > t_lo), so the tensor-core and small-graph kernels keep their launch shape,
// shared memory and results for every other graph.  Correctness, not speed, is the point; the cost is in DESIGN.md §K3.
//
// Element type TE:
//   __nv_bfloat16 — the training path (`precision=16`): bf16 operands and outputs, fp32 math.  The operands the tensor-core
//                   kernels feed their MMAs in bf16 are rounded here the same way: the unnormalised probabilities of P.V,
//                   the (dropped) probabilities of dV = P^T dO, and dS of dQ = dS K and dK = dS^T Q.  t_lo = 513.
//   float         — the fp32 mode's backward for batches whose largest graph has more than 513 tokens (every graph of such a
//                   batch, t_lo = 0): the same arithmetic, in the same order, as k3f_attn_bwd_kernel.
//
// Layout: a CTA works on (plane, chunk of kRows query rows or key columns); its operands are staged in shared memory as fp32
// with an odd row pitch d + 1.  The backward is two kernels, so each stages half of what one pass over both would need:
//   pass A (k3l_bwd_dq_kernel),  warp = query row i, K and V staged: dS row -> dbias, dQ_i = scale * sum_j dS_ij K_j;
//   pass B (k3l_bwd_dkv_kernel), warp = key column j, Q, dO, lse and D staged: dS column recomputed (the same expression,
//          bitwise the same value), dK_j = scale * sum_i dS_ij Q_i, dV_j = sum_i (mask P / keep)_ij dO_i.
// Every sum runs in a fixed order (lanes stride over the other index, d-wide partials merged by shuffles): no atomics,
// bitwise reproducible.  1 025 x (24 + 1) x 2 fp32 = 205 KB of shared memory at most per CTA, one CTA per SM.
// The dropout mask is the tensor-core path's (common.cuh attn_drop_*: same seed, same mask).
#include <cuda_bf16.h>

#include "common.cuh"
#include "k3_small.cuh"

namespace mobgt {

namespace {
constexpr int kLWarps = 8;
constexpr int kLThreads = kLWarps * 32;
constexpr int kRows = 64;   // query rows (forward, pass A) or key columns (pass B) per CTA

__device__ __forceinline__ float to_f(float x) { return x; }
__device__ __forceinline__ float to_f(__nv_bfloat16 x) { return __bfloat162float(x); }
template <typename TE> __device__ __forceinline__ TE from_f(float x);
template <> __device__ __forceinline__ float from_f<float>(float x) { return x; }
template <> __device__ __forceinline__ __nv_bfloat16 from_f<__nv_bfloat16>(float x) { return __float2bfloat16_rn(x); }
// an MMA operand of the tensor-core path: rounded to bf16 in bf16 mode, untouched in fp32 mode
template <typename TE> __device__ __forceinline__ float mma_operand(float x) { return to_f(from_f<TE>(x)); }

__device__ __forceinline__ float lwarp_sum(float x) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xFFFFFFFFu, x, o);
    return x;
}
__device__ __forceinline__ float lwarp_max(float x) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) x = fmaxf(x, __shfl_xor_sync(0xFFFFFFFFu, x, o));
    return x;
}
template <typename TE, int kD>
__device__ __forceinline__ void lstage(const TE *src, int64_t stride, int t0, int Tg, int h, float *dst) {
    for (int i = threadIdx.x; i < Tg * kD; i += kLThreads) {
        const int r = i / kD, e = i - r * kD;
        dst[r * (kD + 1) + e] = to_f(src[(size_t)(t0 + r) * stride + h * kD + e]);
    }
}
template <typename TE, int kD>
__device__ __forceinline__ void lrow(const TE *src, float (&f)[kD]) {
#pragma unroll
    for (int e = 0; e < kD; ++e) f[e] = to_f(src[e]);
}
template <int kD>
__device__ __forceinline__ float ldot(const float (&a)[kD], const float *b) {
    float s = 0.f;
#pragma unroll
    for (int e = 0; e < kD; ++e) s = fmaf(a[e], b[e], s);
    return s;
}
__device__ __forceinline__ bool lkeep(bool on, uint32_t rowkey, int col, uint32_t th16) {
    return !on || ((attn_drop_keep8(rowkey, (uint32_t)(col >> 3), th16) >> (col & 7)) & 1u);
}

// The (graph, head) of CTA row blockIdx.y in launch order and its chunk; false when the graph is not this launch's.
struct LItem { int g, h, plane, t0, Tg, c0, c1; };
__device__ __forceinline__ bool litem(const LargeAttnParams &p, LItem &it) {
    const int gi = blockIdx.y / p.H;
    it.h = blockIdx.y - gi * p.H;
    it.g = p.order ? p.order[gi] : gi;
    it.t0 = p.tok_off[it.g];
    it.Tg = p.tok_off[it.g + 1] - it.t0;
    it.plane = it.g * p.H + it.h;
    it.c0 = blockIdx.x * kRows;
    it.c1 = min(it.c0 + kRows, it.Tg);
    return it.Tg > p.t_lo && it.c0 < it.Tg;
}
}  // namespace

// ---------------------------------------------------------------------------------------------------------------- forward
template <typename TE, int kD>
__global__ void __launch_bounds__(kLThreads) k3l_attn_fwd_kernel(const LargeAttnParams p) {
    constexpr int kPitch = kD + 1;
    extern __shared__ __align__(16) float smem[];
    LItem it;
    if (!litem(p, it)) return;
    const TE *q = static_cast<const TE *>(p.q), *k = static_cast<const TE *>(p.k), *v = static_cast<const TE *>(p.v);
    const TE *bias = static_cast<const TE *>(p.bias);
    TE *out = static_cast<TE *>(p.out);
    float *sK = smem, *sV = smem + it.Tg * kPitch;
    lstage<TE, kD>(k, p.qkv_stride, it.t0, it.Tg, it.h, sK);
    lstage<TE, kD>(v, p.qkv_stride, it.t0, it.Tg, it.h, sV);
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const bool drop = p.drop.th16 != 0;
    uint32_t seed_lo = 0, seed_hi = 0;
    if (drop) attn_drop_fold_seed(p.drop, seed_lo, seed_hi);
    for (int i = it.c0 + warp; i < it.c1; i += kLWarps) {
        float qi[kD];
        lrow<TE, kD>(q + (size_t)(it.t0 + i) * p.qkv_stride + it.h * kD, qi);
        const TE *brow = bias + ((size_t)it.plane * p.T + i) * p.Tp;
        const uint32_t rowkey = drop ? attn_drop_rowkey((uint32_t)it.plane, (uint32_t)i, seed_lo, seed_hi) : 0u;
        float m = -INFINITY;
        for (int j = lane; j < it.Tg; j += 32) m = fmaxf(m, fmaf(p.scale, ldot(qi, sK + j * kPitch), to_f(brow[j])));
        m = lwarp_max(m);
        float l = 0.f, o[kD];
#pragma unroll
        for (int e = 0; e < kD; ++e) o[e] = 0.f;
        for (int j = lane; j < it.Tg; j += 32) {
            const float pe = expf(fmaf(p.scale, ldot(qi, sK + j * kPitch), to_f(brow[j])) - m);
            l += pe;                                          // the denominator is taken before the dropout mask
            if (lkeep(drop, rowkey, j, p.drop.th16)) {
                const float pm = mma_operand<TE>(pe);
                const float *vr = sV + j * kPitch;
#pragma unroll
                for (int e = 0; e < kD; ++e) o[e] = fmaf(pm, vr[e], o[e]);
            }
        }
        l = lwarp_sum(l);
        const float inv = (drop ? p.drop.inv_keep : 1.0f) / l;
        float mine = 0.f;
#pragma unroll
        for (int e = 0; e < kD; ++e) {
            const float s = lwarp_sum(o[e]);
            if (lane == e) mine = s;
        }
        if (lane < kD) out[(size_t)(it.t0 + i) * (p.H * kD) + it.h * kD + lane] = from_f<TE>(mine * inv);
        if (lane == 0) p.lse[(size_t)(it.t0 + i) * p.H + it.h] = m + logf(l);
    }
}

// ---------------------------------------------------------------------------------------------------------------- backward
// D_i = dO_i . O_i, fma chain over e ascending (pass A per row, pass B per staged row: the same value)
template <typename TE, int kD>
__device__ __forceinline__ float ldelta(const LargeAttnParams &p, int t0, int i, int h) {
    const TE *og = static_cast<const TE *>(p.o) + (size_t)(t0 + i) * (p.H * kD) + h * kD;
    const TE *dg = static_cast<const TE *>(p.dout) + (size_t)(t0 + i) * (p.H * kD) + h * kD;
    float d = 0.f;
#pragma unroll
    for (int e = 0; e < kD; ++e) d = fmaf(to_f(og[e]), to_f(dg[e]), d);
    return d;
}

// pass A: warp = query row i
template <typename TE, int kD>
__global__ void __launch_bounds__(kLThreads) k3l_bwd_dq_kernel(const LargeAttnParams p) {
    constexpr int kPitch = kD + 1;
    extern __shared__ __align__(16) float smem[];
    LItem it;
    if (!litem(p, it)) return;
    const TE *q = static_cast<const TE *>(p.q), *k = static_cast<const TE *>(p.k), *v = static_cast<const TE *>(p.v);
    const TE *bias = static_cast<const TE *>(p.bias), *dout = static_cast<const TE *>(p.dout);
    TE *dq = static_cast<TE *>(p.dq);
    float *sK = smem, *sV = smem + it.Tg * kPitch;
    lstage<TE, kD>(k, p.qkv_stride, it.t0, it.Tg, it.h, sK);
    lstage<TE, kD>(v, p.qkv_stride, it.t0, it.Tg, it.h, sV);
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const bool drop = p.drop.th16 != 0;
    const float ik = drop ? p.drop.inv_keep : 1.0f;
    uint32_t seed_lo = 0, seed_hi = 0;
    if (drop) attn_drop_fold_seed(p.drop, seed_lo, seed_hi);
    const size_t pl = (size_t)it.plane * p.T * p.Tp;
    const int HD = p.H * kD;
    for (int i = it.c0 + warp; i < it.c1; i += kLWarps) {
        float qi[kD], dO[kD], dqa[kD];
        lrow<TE, kD>(q + (size_t)(it.t0 + i) * p.qkv_stride + it.h * kD, qi);
        lrow<TE, kD>(dout + (size_t)(it.t0 + i) * HD + it.h * kD, dO);
#pragma unroll
        for (int e = 0; e < kD; ++e) dqa[e] = 0.f;
        const float lse = p.lse[(size_t)(it.t0 + i) * p.H + it.h], del = ldelta<TE, kD>(p, it.t0, i, it.h);
        const uint32_t rowkey = drop ? attn_drop_rowkey((uint32_t)it.plane, (uint32_t)i, seed_lo, seed_hi) : 0u;
        const TE *brow = bias + pl + (size_t)i * p.Tp;
        for (int j = lane; j < it.Tg; j += 32) {
            const float *kr = sK + j * kPitch;
            const float pr = expf(fmaf(p.scale, ldot(qi, kr), to_f(brow[j])) - lse);
            const float dp = lkeep(drop, rowkey, j, p.drop.th16) ? ldot(dO, sV + j * kPitch) * ik : 0.f;
            const float ds = pr * (dp - del);
            const size_t cell = pl + (size_t)i * p.Tp + j;
            if (p.accumulate == 2) {
                static_cast<__nv_bfloat16 *>(p.dbias)[cell] = __float2bfloat16_rn(ds);
            } else {
                float *db = static_cast<float *>(p.dbias) + cell;
                *db = (p.accumulate == 1 ? *db : 0.f) + ds;
            }
            const float dm = mma_operand<TE>(ds);
#pragma unroll
            for (int e = 0; e < kD; ++e) dqa[e] = fmaf(dm, kr[e], dqa[e]);
        }
        float mine = 0.f;
#pragma unroll
        for (int e = 0; e < kD; ++e) {
            const float s = lwarp_sum(dqa[e]);
            if (lane == e) mine = s;
        }
        if (lane < kD) dq[(size_t)(it.t0 + i) * p.dqkv_stride + it.h * kD + lane] = from_f<TE>(mine * p.scale);
    }
}

// pass B: warp = key column j
template <typename TE, int kD>
__global__ void __launch_bounds__(kLThreads) k3l_bwd_dkv_kernel(const LargeAttnParams p) {
    constexpr int kPitch = kD + 1;
    extern __shared__ __align__(16) float smem[];
    LItem it;
    if (!litem(p, it)) return;
    const TE *q = static_cast<const TE *>(p.q), *k = static_cast<const TE *>(p.k), *v = static_cast<const TE *>(p.v);
    const TE *bias = static_cast<const TE *>(p.bias), *dout = static_cast<const TE *>(p.dout);
    TE *dk = static_cast<TE *>(p.dk), *dv = static_cast<TE *>(p.dv);
    const int HD = p.H * kD;
    float *sQ = smem, *sdO = sQ + it.Tg * kPitch, *sLse = sdO + it.Tg * kPitch, *sDel = sLse + it.Tg;
    lstage<TE, kD>(q, p.qkv_stride, it.t0, it.Tg, it.h, sQ);
    lstage<TE, kD>(dout, HD, it.t0, it.Tg, it.h, sdO);
    for (int i = threadIdx.x; i < it.Tg; i += kLThreads) {
        sDel[i] = ldelta<TE, kD>(p, it.t0, i, it.h);
        sLse[i] = p.lse[(size_t)(it.t0 + i) * p.H + it.h];
    }
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const bool drop = p.drop.th16 != 0;
    const float ik = drop ? p.drop.inv_keep : 1.0f;
    uint32_t seed_lo = 0, seed_hi = 0;
    if (drop) attn_drop_fold_seed(p.drop, seed_lo, seed_hi);
    const size_t pl = (size_t)it.plane * p.T * p.Tp;
    for (int j = it.c0 + warp; j < it.c1; j += kLWarps) {
        float kj[kD], vj[kD], dka[kD], dva[kD];
        lrow<TE, kD>(k + (size_t)(it.t0 + j) * p.qkv_stride + it.h * kD, kj);
        lrow<TE, kD>(v + (size_t)(it.t0 + j) * p.qkv_stride + it.h * kD, vj);
#pragma unroll
        for (int e = 0; e < kD; ++e) dka[e] = dva[e] = 0.f;
        for (int i = lane; i < it.Tg; i += 32) {
            const float *qr = sQ + i * kPitch, *dor = sdO + i * kPitch;
            const float pr = expf(fmaf(p.scale, ldot(kj, qr), to_f(bias[pl + (size_t)i * p.Tp + j])) - sLse[i]);
            bool kp = true;
            if (drop) kp = lkeep(true, attn_drop_rowkey((uint32_t)it.plane, (uint32_t)i, seed_lo, seed_hi), j, p.drop.th16);
            const float pd = mma_operand<TE>(kp ? pr * ik : 0.f);
            const float ds = mma_operand<TE>(pr * ((kp ? ldot(vj, dor) * ik : 0.f) - sDel[i]));
#pragma unroll
            for (int e = 0; e < kD; ++e) {
                dka[e] = fmaf(ds, qr[e], dka[e]);
                dva[e] = fmaf(pd, dor[e], dva[e]);
            }
        }
        float mk = 0.f, mv = 0.f;
#pragma unroll
        for (int e = 0; e < kD; ++e) {
            const float a = lwarp_sum(dka[e]), b = lwarp_sum(dva[e]);
            if (lane == e) { mk = a; mv = b; }
        }
        if (lane < kD) {
            dk[(size_t)(it.t0 + j) * p.dqkv_stride + it.h * kD + lane] = from_f<TE>(mk * p.scale);
            dv[(size_t)(it.t0 + j) * p.dqkv_stride + it.h * kD + lane] = from_f<TE>(mv);
        }
    }
}

// ---------------------------------------------------------------------------------------------------------------- launch
// grid: (row chunks of the largest graph, B * H planes in launch order); CTAs of other graphs return at once
template <typename TE, int kD>
int32_t launch_large_attn_fwd(const LargeAttnParams &p, int B, int t_max, cudaStream_t s) {
    const size_t smem = (size_t)2 * t_max * (kD + 1) * sizeof(float);
    auto kern = k3l_attn_fwd_kernel<TE, kD>;
    MOBGT_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<dim3((unsigned)ceil_div(t_max, kRows), (unsigned)(B * p.H)), kLThreads, smem, s>>>(p);
    MOBGT_LAUNCH_OK("k3l_attn_fwd_kernel");
    return MOBGT_OK;
}

template <typename TE, int kD>
int32_t launch_large_attn_bwd(const LargeAttnParams &p, int B, int t_max, cudaStream_t s) {
    const dim3 grid((unsigned)ceil_div(t_max, kRows), (unsigned)(B * p.H));
    const size_t smem_a = (size_t)2 * t_max * (kD + 1) * sizeof(float);                          // K, V
    const size_t smem_b = ((size_t)2 * t_max * (kD + 1) + 2 * (size_t)t_max) * sizeof(float);    // Q, dO, lse, D
    auto ka = k3l_bwd_dq_kernel<TE, kD>;
    auto kb = k3l_bwd_dkv_kernel<TE, kD>;
    MOBGT_CUDA_OK(cudaFuncSetAttribute(ka, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_a));
    MOBGT_CUDA_OK(cudaFuncSetAttribute(kb, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_b));
    ka<<<grid, kLThreads, smem_a, s>>>(p);
    MOBGT_LAUNCH_OK("k3l_bwd_dq_kernel");
    kb<<<grid, kLThreads, smem_b, s>>>(p);
    MOBGT_LAUNCH_OK("k3l_bwd_dkv_kernel");
    return MOBGT_OK;
}

template int32_t launch_large_attn_fwd<__nv_bfloat16, 16>(const LargeAttnParams &, int, int, cudaStream_t);
template int32_t launch_large_attn_fwd<__nv_bfloat16, 24>(const LargeAttnParams &, int, int, cudaStream_t);
template int32_t launch_large_attn_bwd<__nv_bfloat16, 16>(const LargeAttnParams &, int, int, cudaStream_t);
template int32_t launch_large_attn_bwd<__nv_bfloat16, 24>(const LargeAttnParams &, int, int, cudaStream_t);
template int32_t launch_large_attn_bwd<float, 16>(const LargeAttnParams &, int, int, cudaStream_t);
template int32_t launch_large_attn_bwd<float, 24>(const LargeAttnParams &, int, int, cudaStream_t);

}  // namespace mobgt
