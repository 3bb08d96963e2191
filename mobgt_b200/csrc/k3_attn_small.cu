// K3 (small graphs) — the biased attention of model_fqandtoyo.py:1693-1706 and its backward for graphs of at most
// kSmallT = 16 tokens, in plain SIMT fp32 math.
//
// Why: a trajectory graph has 4 nodes in the median (SURVEY.md §8d node-count law; 9 graphs in 10 have at most 16 tokens).  The
// tensor-core kernels (k3_attn_fwd.cu / k3_attn_bwd.cu) spend one CTA, one 128 x 128 MMA tile, a 32 KB TMA bias tile and a
// barrier / TMEM / TMA latency chain of ~20 k cycles on every (graph, head) — for a 5-token graph 99.8 % of that tile is
// padding.  Here a 64-thread CTA (backward: 128 threads, the two passes side by side) works on one graph and four heads,
// thread = (row, head): query row in the forward and in the dQ / dS pass, key column in the dK / dV pass; K, V (and Q, dO in the backward) and the live corner of the bias planes are
// staged once in shared memory (every thread issues its loads back to back: one global-memory latency per CTA), operand rows
// are read as broadcasts, and only the live cells of the dS plane are written.  The arithmetic is the tensor-core path's
// (softmax in log2 units, denominator before the dropout mask, the SAME counter-based mask: common.cuh attn_drop_*), with fp32
// probabilities instead of bf16-rounded MMA operands.
//
// The two paths split the batch on the device: the tensor-core kernels return at once for graphs with Tg <= small_t, these
// kernels for graphs with Tg > small_t, so one CUDA graph captured for a (bucketed) batch shape serves every mix of sizes; the
// entry points launch the two kernels on two streams (fork / join by events, legal inside a capture), since they touch
// disjoint graphs.  Measured on the natural node-count law (256 graphs, 60 000 POIs; profiles/r3/): per layer and direction
// ~22 us for either kernel, overlapped — against 37 us (forward) / 59 us (backward) when every graph took a tensor-core CTA.
// What was tried and dropped: one CTA per (graph, head) with thread = row (5 live lanes in each of 8 warps: 5.7 M issued warp
// instructions per launch), four threads per row with shuffle merges (shorter chains, more instructions), a 64-token threshold
// (the 17..64-token graphs cost more as SIMT than as one more CTA in the tensor-core kernel's single wave).
#include <cuda_bf16.h>

#include "common.cuh"
#include "k3_small.cuh"

namespace mobgt {

namespace {
constexpr float kL2e = 1.4426950408889634f;

__device__ __forceinline__ float ex2(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ void unpack8(const uint4 &a, float *f) {
    const uint32_t w[4] = {a.x, a.y, a.z, a.w};
#pragma unroll
    for (int e = 0; e < 4; ++e) {
        f[2 * e] = __uint_as_float(w[e] << 16);
        f[2 * e + 1] = __uint_as_float(w[e] & 0xFFFF0000u);
    }
}
__device__ __forceinline__ uint32_t pack2(float lo, float hi) {
    __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
    return *reinterpret_cast<uint32_t *>(&v);
}
template <int kD>
__device__ __forceinline__ float dotd(const float (&a)[kD], const float *b) {   // b: shared memory, same address in every lane
    float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;     // four independent chains (a single one is d dependent FMAs)
#pragma unroll
    for (int e = 0; e < kD; e += 4) {
        const float4 v = *reinterpret_cast<const float4 *>(b + e);
        s0 = fmaf(a[e], v.x, s0);
        s1 = fmaf(a[e + 1], v.y, s1);
        s2 = fmaf(a[e + 2], v.z, s2);
        s3 = fmaf(a[e + 3], v.w, s3);
    }
    return (s0 + s1) + (s2 + s3);
}
template <int kD>
__device__ __forceinline__ void axpyd(float (&acc)[kD], float a, const float *b) {
#pragma unroll
    for (int e = 0; e < kD; e += 4) {
        const float4 v = *reinterpret_cast<const float4 *>(b + e);
        acc[e] = fmaf(a, v.x, acc[e]);
        acc[e + 1] = fmaf(a, v.y, acc[e + 1]);
        acc[e + 2] = fmaf(a, v.z, acc[e + 2]);
        acc[e + 3] = fmaf(a, v.w, acc[e + 3]);
    }
}
template <int kD>
__device__ __forceinline__ void stored(__nv_bfloat16 *dst, const float (&a)[kD], float scale) {
    uint4 *d = reinterpret_cast<uint4 *>(dst);
#pragma unroll
    for (int c = 0; c < kD / 8; ++c)
        d[c] = make_uint4(pack2(a[8 * c] * scale, a[8 * c + 1] * scale), pack2(a[8 * c + 2] * scale, a[8 * c + 3] * scale),
                          pack2(a[8 * c + 4] * scale, a[8 * c + 5] * scale), pack2(a[8 * c + 6] * scale, a[8 * c + 7] * scale));
}
}  // namespace

// Thread layout: a CTA of 64 threads works on ONE graph and FOUR heads: tid = 4 * row + head-in-group, row < 16.  All rows of a
// graph share its K / V / Q / dO rows, so one warp covers 8 rows x 4 heads and a 5-token graph keeps 20 lanes of a single warp
// busy (a CTA per (graph, head) would run 5 lanes in each of 8 warps: the kernels are bound by issued instructions).
constexpr int kHG = 4;                                   // heads per CTA
constexpr int kRows = kSmallT;                           // 16
constexpr int kThreads = kHG * kRows;
// operand rows in shared memory: [head-in-group][row][d floats] (+ 4 floats after every 8 rows): the four heads of a warp read
// bank groups 8 apart, the rows of a warp read the same address (broadcast).  A float4 read of a warp is served in phases of
// 8 lanes = 2 rows x 4 heads, i.e. 4 distinct addresses h * kOpFloats + c: conflict-free when kOpFloats mod 32 puts the four
// 4-bank windows apart.  Unpadded, 16 rows x d floats is a multiple of 32 for both head dims (384 and 256: all four heads on
// the same banks); the 2 x 4 floats of padding make it 8 (mod 32) -> windows at banks 0, 8, 16, 24.
template <int kD> __device__ __forceinline__ int row_off(int r) { return r * kD + (r >> 3) * 4; }
template <int kD> constexpr int op_floats() { return kRows * kD + (kRows / 8) * 4; }
static_assert(op_floats<24>() % 32 == 8 && op_floats<16>() % 32 == 8, "d = 24: 392 = 8 (mod 32); d = 16: 264 = 8 (mod 32)");
constexpr int kBP = kRows + 8;                           // bias row pitch (bf16): 48 B, 8 consecutive rows hit distinct banks

// rows [t0, t0 + Tg) x (4 heads x d) bf16 of a [ntok, stride] matrix -> fp32 dst[head][row_off(row)]
template <int kD>
__device__ __forceinline__ void stage_heads(const __nv_bfloat16 *src, int64_t stride, int t0, int Tg, int h0, float *dst, int nthr,
                                            int tid0 = -1) {
    constexpr int kC = kD / 8, kRowC = kHG * kC;         // 16-byte chunks per head / per row slice of the four heads
    for (int i = tid0 < 0 ? (int)threadIdx.x : tid0; i < Tg * kRowC; i += nthr) {
        const int r = i / kRowC, c = i - r * kRowC;      // 16-byte chunk c of the row's 8 d-byte slice: head c / kC, part c % kC
        float f[8];
        unpack8(__ldg(reinterpret_cast<const uint4 *>(src + (size_t)(t0 + r) * stride + h0 * kD) + c), f);
        float4 *d = reinterpret_cast<float4 *>(dst + (c / kC) * op_floats<kD>() + row_off<kD>(r) + (c % kC) * 8);
        d[0] = make_float4(f[0], f[1], f[2], f[3]);
        d[1] = make_float4(f[4], f[5], f[6], f[7]);
    }
}
__device__ __forceinline__ void stage_bias4(const __nv_bfloat16 *bias, int T, int Tp, int plane0, int Tg, __nv_bfloat16 *dst, int nthr,
                                            int tid0 = -1) {
    const int nch = (Tg + 7) >> 3;
    for (int i = tid0 < 0 ? (int)threadIdx.x : tid0; i < kHG * Tg * nch; i += nthr) {
        const int hq = i / (Tg * nch), ii = i - hq * (Tg * nch);
        const int r = ii / nch, c8 = ii - r * nch;
        *reinterpret_cast<uint4 *>(dst + (hq * kRows + r) * kBP + c8 * 8) =
            __ldg(reinterpret_cast<const uint4 *>(bias + ((size_t)(plane0 + hq) * T + r) * Tp) + c8);
    }
}

// ---------------------------------------------------------------------------------------------------------------- forward
template <int kD, bool kDrop>
__global__ void __launch_bounds__(kThreads, 12) k3s_attn_fwd_kernel(const SmallAttnParams p) {
    constexpr int kOpFloats = op_floats<kD>();
    __shared__ __align__(16) float sK[kHG * kOpFloats], sV[kHG * kOpFloats];
    __shared__ __align__(16) __nv_bfloat16 sB[kHG * kRows * kBP];
    const int ngrp = p.H / kHG;
    const int gi = blockIdx.x / ngrp, hg = blockIdx.x - gi * ngrp;
    const int g = p.order ? p.order[gi] : gi;
    const int t0 = p.tok_off[g];
    const int Tg = p.tok_off[g + 1] - t0;
    if (Tg > p.small_t || Tg <= 0) return;                 // the tensor-core kernel's graph
    const int nthr = min(kThreads, kHG * ((Tg + 7) & ~7));  // whole warps (8 rows each) that hold a live row
    if ((int)threadIdx.x >= nthr) return;
    const int h0 = hg * kHG, plane0 = g * p.H + h0;
    stage_bias4(p.bias, p.T, p.Tp, plane0, Tg, sB, nthr);
    stage_heads<kD>(p.k, p.qkv_stride, t0, Tg, h0, sK, nthr);
    stage_heads<kD>(p.v, p.qkv_stride, t0, Tg, h0, sV, nthr);
    const int r = threadIdx.x >> 2, hq = threadIdx.x & 3;
    const bool live = r < Tg;
    const int h = h0 + hq, plane = plane0 + hq;
    const float sl2 = p.scale * kL2e;
    float q[kD];
    if (live) {
        const uint4 *qg = reinterpret_cast<const uint4 *>(p.q + (size_t)(t0 + r) * p.qkv_stride + h * kD);
#pragma unroll
        for (int c = 0; c < kD / 8; ++c) unpack8(__ldg(qg + c), q + 8 * c);
#pragma unroll
        for (int e = 0; e < kD; ++e) q[e] *= sl2;
    }
    asm volatile("bar.sync 1, %0;" ::"r"(nthr) : "memory");   // the live warps (the others have left)
    if (!live) return;
    uint32_t seed_lo = 0, seed_hi = 0;
    if (kDrop) attn_drop_fold_seed(p.drop, seed_lo, seed_hi);
    const uint32_t rowkey = kDrop ? attn_drop_rowkey((uint32_t)plane, (uint32_t)r, seed_lo, seed_hi) : 0u;
    const uint4 *brow = reinterpret_cast<const uint4 *>(sB + (hq * kRows + r) * kBP);
    const float *Kh = sK + hq * kOpFloats, *Vh = sV + hq * kOpFloats;
    float m = -INFINITY, l = 0.f, o[kD];
#pragma unroll
    for (int e = 0; e < kD; ++e) o[e] = 0.f;
    const int nch = (Tg + 7) >> 3;
    for (int c8 = 0; c8 < nch; ++c8) {
        float b8[8], s8[8];
        unpack8(brow[c8], b8);
        const int nv = min(8, Tg - c8 * 8);            // live key columns of this chunk (the rest of the pitch is never written)
        float mc = -INFINITY;
#pragma unroll
        for (int e = 0; e < 8; ++e) {
            s8[e] = -INFINITY;
            if (e < nv) {
                s8[e] = fmaf(b8[e], kL2e, dotd(q, Kh + row_off<kD>(c8 * 8 + e)));
                mc = fmaxf(mc, s8[e]);
            }
        }
        const float m_new = fmaxf(m, mc) == -INFINITY ? 0.f : fmaxf(m, mc);   // (a row of -inf scores stays finite arithmetic)
        const float alpha = ex2(m - m_new);            // first chunk: 2^(-inf) = 0
        l *= alpha;
#pragma unroll
        for (int e = 0; e < kD; ++e) o[e] *= alpha;
        const uint32_t keep = kDrop ? attn_drop_keep8(rowkey, (uint32_t)c8, p.drop.th16) : 0xFFu;
#pragma unroll
        for (int e = 0; e < 8; ++e) {
            if (e < nv) {
                const float pe = ex2(s8[e] - m_new);
                l += pe;                               // the denominator is taken before the dropout mask
                if ((keep >> e) & 1u) axpyd(o, pe, Vh + row_off<kD>(c8 * 8 + e));
            }
        }
        m = m_new;
    }
    stored(p.out + (size_t)(t0 + r) * (p.H * kD) + h * kD, o, (kDrop ? p.drop.inv_keep : 1.0f) / l);
    p.lse[(size_t)(t0 + r) * p.H + h] = (m + log2f(l)) * 0.6931471805599453f;
}

// ---------------------------------------------------------------------------------------------------------------- backward
// pass 1, thread = (query row t, head): D = sum(dO_t * O_t); per key c: p = 2^(s - lse), dP = dO_t . V_c (masked, / keep),
//         dS = p (dP - D) -> dS plane, dQ_t += dS K_c
// pass 2, thread = (key column t, head): the same p / dS recomputed per query row r: dK_t += dS Q_r, dV_t += (mask p / keep) dO_r
// The two passes read the same staged operands and write disjoint outputs, so they run SIDE BY SIDE: threads [0, 64) take
// pass 1, threads [64, 128) pass 2 — the kernel is bound by the dependent-instruction chain of its largest graph, and the
// chain is now the longer of the two passes instead of their sum.
template <int kD, bool kDrop>
__global__ void __launch_bounds__(2 * kThreads, 4) k3s_attn_bwd_kernel(const SmallAttnParams p) {
    constexpr int kOpFloats = op_floats<kD>();
    __shared__ __align__(16) float sQ[kHG * kOpFloats], sK[kHG * kOpFloats], sV[kHG * kOpFloats], sdO[kHG * kOpFloats];
    __shared__ float sLse[kHG * kRows], sDel[kHG * kRows];
    __shared__ __align__(16) __nv_bfloat16 sB[kHG * kRows * kBP];
    const int ngrp = p.H / kHG;
    const int gi = blockIdx.x / ngrp, hg = blockIdx.x - gi * ngrp;
    const int g = p.order ? p.order[gi] : gi;
    const int t0 = p.tok_off[g];
    const int Tg = p.tok_off[g + 1] - t0;
    if (Tg > p.small_t || Tg <= 0) return;                 // the tensor-core kernel's graph
    const int half = (int)threadIdx.x / kThreads, lt = (int)threadIdx.x - half * kThreads;
    const int nhalf = min(kThreads, kHG * ((Tg + 7) & ~7));  // whole warps (8 rows each) that hold a live row, per pass
    if (lt >= nhalf) return;
    const int nthr = 2 * nhalf, sid = half * nhalf + lt;     // compact index of this thread among the live ones
    const int h0 = hg * kHG, plane0 = g * p.H + h0;
    const int HD = p.H * kD;
    stage_bias4(p.bias, p.T, p.Tp, plane0, Tg, sB, nthr, sid);
    stage_heads<kD>(p.q, p.qkv_stride, t0, Tg, h0, sQ, nthr, sid);
    stage_heads<kD>(p.k, p.qkv_stride, t0, Tg, h0, sK, nthr, sid);
    stage_heads<kD>(p.v, p.qkv_stride, t0, Tg, h0, sV, nthr, sid);
    stage_heads<kD>(p.dout, HD, t0, Tg, h0, sdO, nthr, sid);
    const int t = lt >> 2, hq = lt & 3;
    const bool live = t < Tg;
    const int h = h0 + hq, plane = plane0 + hq;
    const float sl2 = p.scale * kL2e;
    const float ik = kDrop ? p.drop.inv_keep : 1.0f;
    uint32_t seed_lo = 0, seed_hi = 0;
    if (kDrop) attn_drop_fold_seed(p.drop, seed_lo, seed_hi);
    if (live && half == 0) {
        const uint4 *og = reinterpret_cast<const uint4 *>(p.o + (size_t)(t0 + t) * HD + h * kD);
        const uint4 *dg = reinterpret_cast<const uint4 *>(p.dout + (size_t)(t0 + t) * HD + h * kD);
        float d = 0.f;
#pragma unroll
        for (int c = 0; c < kD / 8; ++c) {
            float a[8], b[8];
            unpack8(__ldg(og + c), a);
            unpack8(__ldg(dg + c), b);
#pragma unroll
            for (int e = 0; e < 8; ++e) d = fmaf(a[e], b[e], d);
        }
        sDel[hq * kRows + t] = d;
        sLse[hq * kRows + t] = p.lse[(size_t)(t0 + t) * p.H + h] * kL2e;
    }
    asm volatile("bar.sync 1, %0;" ::"r"(nthr) : "memory");
    if (!live) return;
    const size_t pl = (size_t)plane * p.T * p.Tp;
    const int nch = (Tg + 7) >> 3;
    const float *Qh = sQ + hq * kOpFloats, *Kh = sK + hq * kOpFloats, *Vh = sV + hq * kOpFloats, *dOh = sdO + hq * kOpFloats;
    const float *Lh = sLse + hq * kRows, *Dh = sDel + hq * kRows;
    // ---- pass 1: row t
    if (half == 0) {
        float q[kD], dO[kD], dq[kD];
#pragma unroll
        for (int e = 0; e < kD; ++e) {
            q[e] = Qh[row_off<kD>(t) + e] * sl2;
            dO[e] = dOh[row_off<kD>(t) + e];
            dq[e] = 0.f;
        }
        const float lse2 = Lh[t], del = Dh[t];
        const uint32_t rowkey = kDrop ? attn_drop_rowkey((uint32_t)plane, (uint32_t)t, seed_lo, seed_hi) : 0u;
        const uint4 *brow = reinterpret_cast<const uint4 *>(sB + (hq * kRows + t) * kBP);
        for (int c8 = 0; c8 < nch; ++c8) {
            float b8[8], ds8[8];
            unpack8(brow[c8], b8);
            const int nv = min(8, Tg - c8 * 8);
            const uint32_t keep = kDrop ? attn_drop_keep8(rowkey, (uint32_t)c8, p.drop.th16) : 0xFFu;
#pragma unroll
            for (int e = 0; e < 8; ++e) {
                ds8[e] = 0.f;
                if (e < nv) {
                    const float *kc = Kh + row_off<kD>(c8 * 8 + e);
                    const float pr = ex2(fmaf(b8[e], kL2e, dotd(q, kc)) - lse2);
                    const float dp = ((keep >> e) & 1u) ? dotd(dO, Vh + row_off<kD>(c8 * 8 + e)) * ik : 0.f;
                    ds8[e] = pr * (dp - del);
                    axpyd(dq, ds8[e], kc);
                }
            }
            const size_t o = pl + (size_t)t * p.Tp + c8 * 8;
            if (p.accumulate == 2) {
                *reinterpret_cast<uint4 *>(reinterpret_cast<__nv_bfloat16 *>(p.dbias) + o) =
                    make_uint4(pack2(ds8[0], ds8[1]), pack2(ds8[2], ds8[3]), pack2(ds8[4], ds8[5]), pack2(ds8[6], ds8[7]));
            } else {
                float *d32 = reinterpret_cast<float *>(p.dbias) + o;
#pragma unroll
                for (int e = 0; e < 8; ++e)
                    if (e < nv) d32[e] = (p.accumulate == 1 ? d32[e] : 0.f) + ds8[e];
            }
        }
        stored(p.dq + (size_t)(t0 + t) * p.dqkv_stride + h * kD, dq, p.scale);
    }
    // ---- pass 2: column t
    else {
        float k[kD], v[kD], dk[kD], dv[kD];
#pragma unroll
        for (int e = 0; e < kD; ++e) {
            k[e] = Kh[row_off<kD>(t) + e] * sl2;
            v[e] = Vh[row_off<kD>(t) + e];
            dk[e] = dv[e] = 0.f;
        }
        const __nv_bfloat16 *bcol = sB + hq * kRows * kBP + t;
        for (int r = 0; r < Tg; ++r) {
            const float *qr = Qh + row_off<kD>(r), *dor = dOh + row_off<kD>(r);
            const float pr = ex2(fmaf(__bfloat162float(bcol[r * kBP]), kL2e, dotd(k, qr)) - Lh[r]);
            bool kp = true;
            if (kDrop) {
                const uint32_t rowkey = attn_drop_rowkey((uint32_t)plane, (uint32_t)r, seed_lo, seed_hi);
                kp = (attn_drop_keep8(rowkey, (uint32_t)(t >> 3), p.drop.th16) >> (t & 7)) & 1u;
            }
            const float pd = kp ? pr * ik : 0.f;
            const float ds = pr * ((kp ? dotd(v, dor) * ik : 0.f) - Dh[r]);
            axpyd(dk, ds, qr);
            axpyd(dv, pd, dor);
        }
        stored(p.dk + (size_t)(t0 + t) * p.dqkv_stride + h * kD, dk, p.scale);
        stored(p.dv + (size_t)(t0 + t) * p.dqkv_stride + h * kD, dv, 1.0f);
    }
}

template <int kD>
int32_t launch_small_attn_fwd(const SmallAttnParams &p, int B, cudaStream_t s) {
    const int grid = B * (p.H / kHG);
    if (p.drop.th16) k3s_attn_fwd_kernel<kD, true><<<grid, kThreads, 0, s>>>(p);
    else k3s_attn_fwd_kernel<kD, false><<<grid, kThreads, 0, s>>>(p);
    MOBGT_LAUNCH_OK("k3s_attn_fwd_kernel");
    return MOBGT_OK;
}

template <int kD>
int32_t launch_small_attn_bwd(const SmallAttnParams &p, int B, cudaStream_t s) {
    const int grid = B * (p.H / kHG);
    if (p.drop.th16) k3s_attn_bwd_kernel<kD, true><<<grid, 2 * kThreads, 0, s>>>(p);
    else k3s_attn_bwd_kernel<kD, false><<<grid, 2 * kThreads, 0, s>>>(p);
    MOBGT_LAUNCH_OK("k3s_attn_bwd_kernel");
    return MOBGT_OK;
}

template int32_t launch_small_attn_fwd<16>(const SmallAttnParams &, int, cudaStream_t);
template int32_t launch_small_attn_fwd<24>(const SmallAttnParams &, int, cudaStream_t);
template int32_t launch_small_attn_bwd<16>(const SmallAttnParams &, int, cudaStream_t);
template int32_t launch_small_attn_bwd<24>(const SmallAttnParams &, int, cudaStream_t);

}  // namespace mobgt
