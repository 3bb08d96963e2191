// K2 — attention-bias build, forward and backward (sm_100a, HBM-bound).
//
// Replaces model_fqandtoyo.py:1143-1216 (fp32 statement: model.py:126-190): the
// rel_pos_encoder / poi_pos_encoder gathers, the graph-token virtual distance, and the multi-hop
// edge encoding (edge_encoder gather along each path, per-hop edge_dis_encoder 8x8 dot, sum over
// hops divided by the clamped path length) fused into ONE pass that reads the compact packed
// indices (i16 rel_pos, i16 poi_pos, u8 edge_input[hops]) and writes bias[B,H,T,Tp].
//
//   bias[g,h,a,b] = [a>=1, b>=1] ( R[rp[g,a-1,b-1],h] + Ppos[pp[g,a-1,b-1],h] + Edge[g,h,a-1,b-1] )
//                 + [a>=1, b==0] t[h]            (row 0 gets no bias: model_fqandtoyo.py:1160-1165)
//   Edge[g,h,i,j] = ( sum_k sum_h' E[ei[g,i,j,k],h'] * W[k,h',h] ) / sp,   sp = clamp(M,1,hops) with M = rp-1
//   (and -inf where M >= rel_pos_max, collator.py:354-358; padding columns are masked inside the
//    attention kernel from seqlens, so the 2*attn_bias term of :1144/:1216 needs no storage).
//
// The 8x8 dot is hoisted out of the pair loop: EW[k][v][h] = sum_h' E[v,h'] W[k,h',h] is a
// [hops,128,H] table (80 KB fp32 at hops=20,H=8) built by a prologue kernel and staged in shared
// memory, so the per-pair work is `walk length` 32-byte shared-memory gathers.  E[0] is a padding row
// (nn.Embedding(padding_idx=0), model_fqandtoyo.py:784) and is structurally zero, so the hop loop stops
// at the first ei == 0.
//
// Backward: dBias (fp32, summed over layers) -> dR, dPpos, dt and dEW by shared-memory-privatised
// histograms (persistent CTAs), then dE = dEW . W^T and dW = E^T . dEW in an epilogue kernel.
#include <cuda_bf16.h>

#include "common.cuh"

namespace mobgt {

// Head counts: every kernel takes H as a template parameter, built for 8 (two float4s per table row) and 12 (three float4s);
// other head counts are UNSUPPORTED.  The tables are [rows][H] fp32, so a row is H / 4 16-byte words.
constexpr int kEdgeVocab = 128;  // edge_encoder rows (model_fqandtoyo.py:784)

struct K2Common {
    const int32_t *n;        // [B]
    const int64_t *sq_off;   // [B+1]
    const int16_t *rel_pos;  // packed [sum n^2]  (M+1)
    const int16_t *poi_pos;  // packed [sum n^2]
    const uint8_t *edge_in;  // packed [sum n^2, hops]  (e+1)
    int B, T, Tp, hops, rel_pos_max;
    int dk;                  // multi_hop_max_dist: walk bytes [dk, hops) are padding (0); sp = clamp(M, 1, dk)
};

constexpr int kDomEdge = 4;    // edge count 1 -> attn_edge_type 3 (wrapper.py:49-53) -> +1 (collator.py:86-93): "one transition"
constexpr int kRelRows = 512;  // rel_pos_encoder rows (model_fqandtoyo.py:786): keys 0..511

// walk length the distance key rp = M + 1 predicts: min(M, hops) for a reachable off-diagonal pair, else 0
__host__ __device__ __forceinline__ int expected_walk(int rp, int hops) {
    const int M = rp - 1;
    return (M < 510) ? min(max(M, 0), hops) : 0;
}

// Prologue tables (workspace):
//   EW[k][v][h] = sum_h' E[v][h'] * W[k][h'][h]                                            [hops][128][H]
//   RL[rp][h]   = R[rp][h] + ( sum_{k < L(rp)} EW[k][dom][h] ) / clamp(rp-1, 1, hops)       [512][H]
// RL is the whole rel_pos-keyed part of the bias of a pair whose walk is the EXPECTED one: L(rp) hops that all carry the
// dominant edge feature (a single transition).  -inf where rp-1 >= rel_pos_max (collator.py:354-358).
template <int H>
__global__ void k2_prep_kernel(const float *__restrict__ E, const float *__restrict__ W, const float *__restrict__ R, int hops,
                               int dk, int rel_pos_max, float *__restrict__ EW, float *__restrict__ RL) {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    const int nEW = hops * kEdgeVocab * H;
    if (idx < nEW) {
        const int h = idx % H, v = (idx / H) % kEdgeVocab, k = idx / (H * kEdgeVocab);
        float acc = 0.f;
#pragma unroll
        for (int hp = 0; hp < H; ++hp) acc += E[v * H + hp] * W[(k * H + hp) * H + h];
        EW[idx] = acc;
    } else if (idx < nEW + kRelRows * H) {
        const int j = idx - nEW;
        const int h = j % H, rp = j / H;
        const int L = expected_walk(rp, dk);
        float ps = 0.f;
        for (int k = 0; k < L; ++k) {
            float acc = 0.f;
#pragma unroll
            for (int hp = 0; hp < H; ++hp) acc += E[kDomEdge * H + hp] * W[(k * H + hp) * H + h];
            ps += acc;
        }
        const int M = rp - 1;
        const float inv = 1.0f / (float)min(max(M, 1), dk);
        RL[j] = (M >= rel_pos_max) ? -INFINITY : R[j] + ps * inv;
    }
}

// one H-float table row as H / 4 float4 loads, all issued before the first is used
template <int H>
__device__ __forceinline__ void load_row(float4 (&x)[H / 4], const float *__restrict__ p) {
#pragma unroll
    for (int i = 0; i < H / 4; ++i) x[i] = *reinterpret_cast<const float4 *>(p + 4 * i);
}
// a[h] += p[h] / a[h] -= p[h] over one table row
template <int H>
__device__ __forceinline__ void add_row(float (&a)[H], const float *__restrict__ p) {
    float4 x[H / 4];
    load_row<H>(x, p);
#pragma unroll
    for (int i = 0; i < H / 4; ++i) {
        a[4 * i] += x[i].x; a[4 * i + 1] += x[i].y; a[4 * i + 2] += x[i].z; a[4 * i + 3] += x[i].w;
    }
}
template <int H>
__device__ __forceinline__ void sub_row(float (&a)[H], const float *__restrict__ p) {
    float4 x[H / 4];
    load_row<H>(x, p);
#pragma unroll
    for (int i = 0; i < H / 4; ++i) {
        a[4 * i] -= x[i].x; a[4 * i + 1] -= x[i].y; a[4 * i + 2] -= x[i].z; a[4 * i + 3] -= x[i].w;
    }
}

// i % H and i / H of a non-negative index (8 heads: the mask and shift the 8-head kernels were written with)
template <int H>
__device__ __forceinline__ int mod_h(int i) {
    if constexpr (H == 8) return i & 7;
    else return (int)((uint32_t)i % H);
}
template <int H>
__device__ __forceinline__ int div_h(int i) {
    if constexpr (H == 8) return i >> 3;
    else return (int)((uint32_t)i / H);
}

__device__ __forceinline__ float bf16lo(uint32_t w) { return __uint_as_float(w << 16); }

template <typename OutT>
__device__ __forceinline__ void store2(OutT *p, float a, float b);
template <>
__device__ __forceinline__ void store2<float>(float *p, float a, float b) { *reinterpret_cast<float2 *>(p) = make_float2(a, b); }
template <>
__device__ __forceinline__ void store2<__nv_bfloat16>(__nv_bfloat16 *p, float a, float b) {
    *reinterpret_cast<__nv_bfloat162 *>(p) = __floats2bfloat162_rn(a, b);
}
template <typename OutT>
__device__ __forceinline__ void store1(OutT *p, float a);
template <>
__device__ __forceinline__ void store1<float>(float *p, float a) { *p = a; }
template <>
__device__ __forceinline__ void store1<__nv_bfloat16>(__nv_bfloat16 *p, float a) { *p = __float2bfloat16_rn(a); }

// expected walk bytes of a pair with walk length L: word q = dominant feature in bytes [4q, 4q+4) ∩ [0, L)
__device__ __forceinline__ uint32_t expected_word(int L, int q) {
    const int r = min(max(L - 4 * q, 0), 4);
    const uint32_t mask = r >= 4 ? 0xFFFFFFFFu : ((1u << (8 * r)) - 1u);
    return (0x01010101u * (uint32_t)kDomEdge) & mask;
}

// cells per forward thread (see the forward's comment)
template <int H>
struct K2FwdCells {
    static constexpr int kCells = H == 8 ? 2 : 1;
};

// Forward.  Persistent CTAs; RL [512][H], Ppos [bins][H] and the expected-walk words XW [hops+1][8] are staged once per
// CTA in shared memory.  At 8 heads, one thread per PAIR OF ADJACENT CELLS (a, b) (a, b+1), b even, of the Tp-pitched
// plane row, so every head plane is written as 4-byte (bf16x2) / 8-byte (f32x2) words and a warp covers 64 consecutive
// columns.  All index bytes of a thread's cells (2 + 2 + hops B each) are fetched up front as independent loads.
// At 12 heads a thread takes ONE cell (K2FwdCells): two cells would keep 2 x 12 accumulators, the correction row and up to
// 2 x 8 walk words live under the 64 registers __launch_bounds__(512, 2) leaves, and spill 32-88 bytes of stack per thread
// (56 at hops = 20).  With one cell the spill is 8 bytes at hops 12..24 and 16 / 24 at hops 28 / 32, no more than the
// 8-head kernel's.  A warp then covers 32 consecutive columns with 2-byte (bf16) / 4-byte (f32) stores.
//
// Per cell the work is TWO table gathers: bias = RL[rp] + Ppos[pp].  The walk bytes are only compared (XOR) against the
// walk the distance predicts; the bytes that differ — another edge feature (0.7 % of the hops of trajectory graphs) or a
// walk cut short by the reference's node-0 quirk (algos.pyx:57-62) — are corrected one by one from the EW table in
// global memory (L1-resident):   Edge = sum_k EW[k][e_k]  =  PS[L] + sum_{k : e_k != x_k} ( EW[k][e_k] - EW[k][x_k] ).
// The identity holds for ANY byte pattern (EW[k][0] = 0: edge_encoder row 0 is the padding row, model_fqandtoyo.py:784).
template <int H, typename OutT, int HOPW>
__global__ void __launch_bounds__(512, 2) k2_bias_fwd_kernel(const K2Common c, const float *__restrict__ RLg,
                                                             const float *__restrict__ Pg, int num_bins,
                                                             const float *__restrict__ tvd,
                                                             const float *__restrict__ EWg, OutT *__restrict__ out) {
    extern __shared__ __align__(16) float sm[];
    const int nR = kRelRows * H, nP = num_bins * H;
    float *RL = sm, *Pp = RL + nR;
    uint32_t *XW = reinterpret_cast<uint32_t *>(Pp + nP);          // [hops + 1][8]
    for (int i = threadIdx.x * 4; i < nR; i += blockDim.x * 4)
        *reinterpret_cast<float4 *>(RL + i) = *reinterpret_cast<const float4 *>(RLg + i);
    for (int i = threadIdx.x * 4; i < nP; i += blockDim.x * 4)
        *reinterpret_cast<float4 *>(Pp + i) = *reinterpret_cast<const float4 *>(Pg + i);
    constexpr int hopw = HOPW;                    // hops = 4 * HOPW
    for (int i = threadIdx.x; i < (c.hops + 1) * 8; i += blockDim.x) XW[i] = (i & 7) < hopw ? expected_word(i >> 3, i & 7) : 0u;
    __syncthreads();
    constexpr int kCells = K2FwdCells<H>::kCells;
    const int half = c.Tp >> (kCells - 1);        // threads per plane row (cell pairs at 8 heads, cells at 12)
    const int per_graph = c.T * half;
    const int tiles = ceil_div(per_graph, (int)blockDim.x);
    const uint64_t half_magic = ((1ull << 40) + half - 1) / half;     // f / half == (f * magic) >> 40 for f < 2^40 / half (> 2^30)
    const size_t hs = (size_t)c.T * c.Tp;
    for (int w = blockIdx.x; w < tiles * c.B; w += gridDim.x) {
        const int g = w / tiles, tile = w - g * tiles;
        const int n = c.n[g];
        const int Tg = n + 1;
        const int f = tile * blockDim.x + threadIdx.x;
        const int a = (int)(((uint64_t)f * half_magic) >> 40), b = (f - a * half) * kCells;
        if (a >= Tg || b >= Tg) continue;
        const bool two = kCells == 2 && b + 1 < Tg;
        float acc[kCells][H];
#pragma unroll
        for (int s = 0; s < kCells; ++s)
#pragma unroll
            for (int h = 0; h < H; ++h) acc[s][h] = 0.f;
        if (a >= 1) {
            const int64_t rowp = c.sq_off[g] + (int64_t)(a - 1) * n;   // pair (a-1, j) lives at rowp + j
            // cell s of this thread is the pair j = b - 1 + s  (b == 0, s == 0: the virtual-distance column)
            int rp[kCells], pp[kCells];
            uint32_t ew[kCells][HOPW];
            bool is_pair[kCells];
#pragma unroll
            for (int s = 0; s < kCells; ++s) {
                const int j = b - 1 + s;
                is_pair[s] = j >= 0 && j < n;
                rp[s] = 0; pp[s] = 0;
#pragma unroll
                for (int q = 0; q < HOPW; ++q) ew[s][q] = 0u;
                if (is_pair[s]) {
                    const int64_t pc = rowp + j;
                    rp[s] = c.rel_pos[pc];
                    pp[s] = c.poi_pos[pc];
                    const uint32_t *ei = reinterpret_cast<const uint32_t *>(c.edge_in + pc * c.hops);
#pragma unroll
                    for (int q = 0; q < HOPW; ++q) ew[s][q] = __ldg(ei + q);
                }
            }
#pragma unroll
            for (int s = 0; s < kCells; ++s) {
                if (!is_pair[s]) {
                    if (b == 0 && s == 0) {
#pragma unroll
                        for (int h = 0; h < H; ++h) acc[0][h] = __ldg(tvd + h);
                    }
                    continue;
                }
                const int rk = min(max(rp[s], 0), kRelRows - 1);
                const int L = expected_walk(rk, c.dk);
                const uint4 x0 = *reinterpret_cast<const uint4 *>(XW + L * 8), x1 = *reinterpret_cast<const uint4 *>(XW + L * 8 + 4);
                const uint32_t xw[8] = {x0.x, x0.y, x0.z, x0.w, x1.x, x1.y, x1.z, x1.w};
                uint32_t any = 0u;
#pragma unroll
                for (int q = 0; q < HOPW; ++q) any |= ew[s][q] ^ xw[q];
                const float *r = RL + rk * H, *q_ = Pp + min(max(pp[s], 0), num_bins - 1) * H;
                float4 r0[H / 4], p0[H / 4];
                load_row<H>(r0, r);
                load_row<H>(p0, q_);
#pragma unroll
                for (int i = 0; i < H / 4; ++i) {
                    acc[s][4 * i] = r0[i].x + p0[i].x; acc[s][4 * i + 1] = r0[i].y + p0[i].y;
                    acc[s][4 * i + 2] = r0[i].z + p0[i].z; acc[s][4 * i + 3] = r0[i].w + p0[i].w;
                }
                if (any != 0u) {
                    float corr[H] = {};
#pragma unroll
                    for (int q = 0; q < HOPW; ++q) {
                        {
                            uint32_t d = ew[s][q] ^ xw[q];
                            while (d != 0u) {
                                const int e = (__ffs(d) - 1) >> 3;
                                const int v = (ew[s][q] >> (8 * e)) & 0xFF, x = (xw[q] >> (8 * e)) & 0xFF;
                                const float *row = EWg + (size_t)(q * 4 + e) * kEdgeVocab * H;
                                add_row<H>(corr, row + min(v, kEdgeVocab - 1) * H);
                                sub_row<H>(corr, row + x * H);
                                d &= ~(0xFFu << (8 * e));
                            }
                        }
                    }
                    const float inv = 1.0f / (float)min(max(rk - 1, 1), c.dk);
#pragma unroll
                    for (int h = 0; h < H; ++h) acc[s][h] += corr[h] * inv;
                }
            }
        }
        OutT *o = out + ((size_t)g * H * c.T + a) * c.Tp + b;
        if (two) {
#pragma unroll
            for (int h = 0; h < H; ++h) store2<OutT>(o + h * hs, acc[0][h], acc[kCells - 1][h]);
        } else {
#pragma unroll
            for (int h = 0; h < H; ++h) store1<OutT>(o + h * hs, acc[0][h]);
        }
    }
}

// ---- backward --------------------------------------------------------------------------------------
// dBias (per-layer bf16 dS planes, or one fp32 buffer) -> table gradients.  With the forward's decomposition
//   bias(cell) = RL[rp] + Ppos[pp] + ( sum over the bytes that deviate from the expected walk ) / sp
// every cell contributes its H-vector d[h] to exactly TWO keyed sums, dRL[rp] and dPpos[pp] (plus dt for column 0); only
// the deviating bytes (0.09 per cell on trajectory graphs) touch dEW directly.  The finish kernels unfold dRL:
//   dR[rp] = dRL[rp] ;   dEW[k][dom] += sum_{rp : L(rp) > k} dRL[rp] / sp(rp).
// One WARP per plane row (g, a), 1 persistent CTA per SM, three phases per row:
//   1. sum phase   — the row of every (layer, head) plane is read with 16-byte loads (lane = 8-cell chunk of one head, all
//                    layers in flight together), summed in fp32 and parked in the warp's shared-memory strip dsum[h][b];
//   2. index phase — lane = cell: rel_pos, poi_pos and the walk words are read once and packed into cinfo[b] (histogram
//                    rows + flags) and cdev[b] (up to two deviating bytes, so the histogram phase never touches global
//                    memory);
//   3. histogram   — lanes = (table: R | P) x (cell slot) x (head) (K2Heads below): ONE read-modify-write per lane and
//                    step into warp-private histograms laid out [key][cell slot][head] — no atomics, no cross-lane
//                    hazards; two steps are in flight per lane (equal keys are merged in registers).
//   Deviating bytes (the rare path): 64-bit FIXED-POINT integer atomics (value * 2^38) into the CTA's own small dEW table in
//   global memory (features < 16) or into the launch-wide table (other features, rel_pos keys outside the plan).  Integer
//   addition is associative, so the sums do not depend on the order in which the atomics land.
// Per-CTA totals go to a partial buffer and are reduced in a fixed order: the whole backward is bitwise reproducible.
constexpr int kSmallVocab = 16;   // edge features kept in the CTA's shared dEW table

// Lane maps of the backward.  In the histogram phase every lane owns one (table, cell slot, head) column of the warp's
// histograms, so no two lanes ever write the same word, and each step a lane adds two adjacent cells of its slot.
//   H = 8:  2 tables x 2 cell slots x 8 heads = 32 lanes; a step covers 4 cells.
//   H = 12: 2 tables x 12 heads = 24 columns already; a second cell slot would need 48 lanes.  So there is one cell slot, a
//           step covers 2 cells and lanes 24..31 sit the phase out (75 % of the lanes busy).  Splitting the heads over two
//           passes instead (8 + 4 heads, 2 cell slots each) keeps the same 96 read-modify-writes per 64 lane-steps, with
//           a second pass over cinfo; one slot also halves the histograms' shared memory, which buys warps per CTA.
// The slow path gives each listed cell H lanes (one per head): 32 / H cells at a time (4 at H = 8, 2 at H = 12).
template <int H>
struct K2Heads {
    static_assert(H == 8 || H == 12, "the attention-bias kernels are built for 8 and 12 heads");
    static constexpr int kSlots = 32 / (2 * H);       // histogram cell slots
    static constexpr int kLanes = 2 * kSlots * H;     // lanes that own a histogram column
    static constexpr int kSlowCells = 32 / H;         // slow-path cells per round
};

// 12 warps at most: 384 threads leave 170 registers per thread, which the sum phase (18 x 16-byte loads in flight per lane)
// and the index phase (the indices of up to 160 cells of the row loaded before any is decoded) are sized for
constexpr int kK2BwdMaxWarps = 12;
constexpr int kSumItems = 3;     // 16-byte chunks per lane and round of the sum phase
constexpr int kIdxUnroll = 5;    // 32-cell groups whose index loads are issued together

struct K2BwdPlan {
    int Rrows;      // rel_pos histogram rows: keys 0..Rrows-2 direct, key 511 -> row Rrows-1
    int nEWs, nR, nP, stride;   // floats; partial row = [EWsmall | R | P | t(H)]
    int pitch;      // floats per head in the dsum strip: >= T rounded up to 4, == 4 (mod 32)
    int per_warp;   // floats of warp-private shared memory
    int cta_words;  // floats of CTA-wide shared memory in front of the warp strips
    int warps;
};

template <int H>
__host__ __device__ inline K2BwdPlan k2_bwd_plan(int T, int Tp, int hops, int num_bins) {
    constexpr int S = K2Heads<H>::kSlots;
    K2BwdPlan p;
    p.Rrows = min(T, 511) + 1;
    p.nEWs = hops * kSmallVocab * H;
    p.nR = p.Rrows * H;
    p.nP = num_bins * H;
    p.stride = p.nEWs + p.nR + p.nP + H;
    // cells b < (T + 3) & ~3 are the ones the index / histogram phases touch; the sum phase clips its 8-cell stores at the pitch
    (void)Tp;
    p.pitch = ((((T + 3) & ~3) + 27) / 32) * 32 + 4;
    p.per_warp = S * (p.nR + H) + S * (p.nP + H) + H * p.pitch + 3 * p.pitch + H;   // hR+trash | hP+trash | dsum | cinfo | cdev | dlist | t
    p.cta_words = (hops + 1) * 8 + 40;                                     // XW | 1/sp table
    int w = (int)((227 * 1024 - 2048 - p.cta_words * 4) / (p.per_warp * 4));
    p.warps = w > kK2BwdMaxWarps ? kK2BwdMaxWarps : w;
    return p;
}

// rare-path accumulators: signed 64-bit fixed point, 38 fractional bits (resolution 3.6e-12, range +-3.3e7)
constexpr double kFxScale = 274877906944.0, kFxInv = 1.0 / 274877906944.0;
__device__ __forceinline__ void fx_add(long long *dst, float v) {
    atomicAdd(reinterpret_cast<unsigned long long *>(dst), (unsigned long long)__double2ll_rn((double)v * kFxScale));
}
__device__ __forceinline__ float fx_to_float(long long v) { return (float)((double)v * kFxInv); }

constexpr uint32_t kInfoPair = 1u << 21, kInfoDev = 1u << 20, kInfoCol0 = 1u << 22, kInfoOvf = 1u << 23, kInfoUnreach = 1u << 24;

__device__ __forceinline__ float lds_f32(uint32_t a) {
    float v;
    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(a) : "memory");
    return v;
}
__device__ __forceinline__ uint32_t lds_u32(uint32_t a) {
    uint32_t v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a) : "memory");
    return v;
}
__device__ __forceinline__ void sts_f32(uint32_t a, float v) { asm volatile("st.shared.f32 [%0], %1;" ::"r"(a), "f"(v) : "memory"); }
__device__ __forceinline__ void sts_u32(uint32_t a, uint32_t v) { asm volatile("st.shared.u32 [%0], %1;" ::"r"(a), "r"(v) : "memory"); }
__device__ __forceinline__ void sts_f32x4(uint32_t a, float x, float y, float z, float w) {
    asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(a), "f"(x), "f"(y), "f"(z), "f"(w) : "memory");
}

// Sum phase of one plane row (g, a) of the backward: dsum[h][b] = sum over layers of plane[l][g][h][a][b] for b < Tg, into the
// warp's shared-memory strip (row pitch `pitch` floats).  The lanes take 16-byte chunks of the row (lane = 8-cell chunk of one
// head), all layers of a chunk in flight together.
template <int H, typename DT>
__device__ __forceinline__ void k2_bwd_sum_row(const DT *__restrict__ rowbase, int Tg, int nlayers, int64_t layer_stride, size_t hs,
                                               uint32_t s_dsum, uint32_t pitch4, int pitch, int lane) {
    constexpr int kPer = 16 / (int)sizeof(DT);           // cells per 16-byte load
    const int nitems = ceil_div(Tg, kPer) * H;           // item i = (chunk i / H, head i % H)
    for (int i0 = 0; i0 < nitems; i0 += 32 * kSumItems) {
        const int ns = min(kSumItems, (nitems - i0 + 31) >> 5);   // 32-item slots of this round that hold an item (warp-uniform)
        float accv[kSumItems][8];
#pragma unroll
        for (int s = 0; s < kSumItems; ++s)
#pragma unroll
            for (int q = 0; q < 8; ++q) accv[s][q] = 0.f;
        const DT *src[kSumItems];
        bool ok[kSumItems];
#pragma unroll
        for (int s = 0; s < kSumItems; ++s) {
            const int i = i0 + 32 * s + lane;
            ok[s] = i < nitems;
            const int ic = min(i, nitems - 1);           // lanes past the last item re-read it (no predicate on the loads)
            src[s] = rowbase + (size_t)mod_h<H>(ic) * hs + div_h<H>(ic) * kPer;
        }
        for (int l0 = 0; l0 < nlayers; l0 += 6) {
            uint4 v[kSumItems][6];
            if (l0 + 6 <= nlayers) {
#pragma unroll
                for (int s = 0; s < kSumItems; ++s)
                    if (s < ns) {
                        const DT *pl0 = src[s] + (size_t)l0 * layer_stride;
#pragma unroll
                        for (int j = 0; j < 6; ++j) v[s][j] = __ldg(reinterpret_cast<const uint4 *>(pl0 + (size_t)j * layer_stride));
                    }
            } else {
#pragma unroll
                for (int s = 0; s < kSumItems; ++s)
                    if (s < ns) {
#pragma unroll
                        for (int j = 0; j < 6; ++j)
                            v[s][j] = (l0 + j < nlayers)
                                          ? __ldg(reinterpret_cast<const uint4 *>(src[s] + (size_t)(l0 + j) * layer_stride))
                                          : make_uint4(0u, 0u, 0u, 0u);
                    }
            }
#pragma unroll
            for (int s = 0; s < kSumItems; ++s)
                if (s < ns) {
#pragma unroll
                    for (int j = 0; j < 6; ++j) {
                        const uint32_t w4[4] = {v[s][j].x, v[s][j].y, v[s][j].z, v[s][j].w};
                        if constexpr (sizeof(DT) == 4) {
#pragma unroll
                            for (int q = 0; q < 4; ++q) accv[s][q] += __uint_as_float(w4[q]);
                        } else {
#pragma unroll
                            for (int q = 0; q < 4; ++q) {
                                accv[s][2 * q] += bf16lo(w4[q]);
                                accv[s][2 * q + 1] += __uint_as_float(w4[q] & 0xFFFF0000u);
                            }
                        }
                    }
                }
        }
#pragma unroll
        for (int s = 0; s < kSumItems; ++s) {
            const int i = i0 + 32 * s + lane;
            if (ok[s]) {
                const uint32_t dst = s_dsum + (uint32_t)mod_h<H>(i) * pitch4 + (uint32_t)(div_h<H>(i) * kPer) * 4u;
                sts_f32x4(dst, accv[s][0], accv[s][1], accv[s][2], accv[s][3]);
                if constexpr (sizeof(DT) == 2) {         // cells past the pitch lie beyond the graph's last token: never read
                    if (div_h<H>(i) * kPer + 8 <= pitch) sts_f32x4(dst + 16u, accv[s][4], accv[s][5], accv[s][6], accv[s][7]);
                }
            }
        }
    }
}

// Histogram phase of one plane row: lane = (table, cell slot c2, head h) adds dsum[h][b] of adjacent cells b0 + 2 c2,
// b0 + 2 c2 + 1 per step into the row of its table that cinfo[b] names (R row in the low 16 bits, P row in the high 16).
// Cells without a gradient point at the trash rows, so the loop carries no predicates.
template <int H>
__device__ __forceinline__ void k2_bwd_hist_row(uint32_t s_cinfo, uint32_t s_dsum, uint32_t s_hist, uint32_t key_shift,
                                                uint32_t pitch4, int Tg4, int lane, int c2, int h) {
    constexpr int S = K2Heads<H>::kSlots;
    constexpr uint32_t key_bytes = S * H * 4;
    if (K2Heads<H>::kLanes == 32 || lane < K2Heads<H>::kLanes) {
        uint32_t pi = s_cinfo + (uint32_t)c2 * 8u, pd = s_dsum + (uint32_t)h * pitch4 + (uint32_t)c2 * 8u;
        for (int b0 = 0; b0 < Tg4; b0 += 2 * S, pi += 8u * S, pd += 8u * S) {
            uint32_t iA, iB;
            float dA, dB_;
            asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(iA), "=r"(iB) : "r"(pi) : "memory");
            asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(dA), "=f"(dB_) : "r"(pd) : "memory");
            const uint32_t aA = s_hist + ((iA >> key_shift) & 0xFFFFu) * key_bytes;
            const uint32_t aB = s_hist + ((iB >> key_shift) & 0xFFFFu) * key_bytes;
            // two read-modify-writes in flight; equal addresses are chained in registers, the second store wins
            const float vA = lds_f32(aA), vB = lds_f32(aB);
            const float nA = vA + dA;
            const float nB = ((aA == aB) ? nA : vB) + dB_;
            sts_f32(aA, nA);
            sts_f32(aB, nB);
        }
    }
}

template <int H, typename DT, int HOPW>
__global__ void __launch_bounds__(kK2BwdMaxWarps * 32, 1) k2_bias_bwd_kernel(const K2Common c, const DT *__restrict__ dB, int nlayers,
                                                             int64_t layer_stride, int num_bins,
                                                             const K2BwdPlan pl, float *__restrict__ partial,
                                                             long long *__restrict__ ews64, long long *__restrict__ dEWfull64,
                                                             long long *__restrict__ dR64) {
    extern __shared__ __align__(16) float sm[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = blockDim.x >> 5;
    constexpr int S = K2Heads<H>::kSlots;
    const int ty = lane / (S * H), c2 = (lane / H) % S, h = lane % H;      // table (0 = R, 1 = P), cell slot, head
    long long *sEW = ews64 + (size_t)blockIdx.x * pl.nEWs;        // this CTA's [hops][16][H] table (global memory, zeroed by the host)
    uint32_t *XW = reinterpret_cast<uint32_t *>(sm);              // [hops + 1][8]
    float *invT = sm + (c.hops + 1) * 8;                          // [40]: 1 / sp
    float *wbase = sm + pl.cta_words;
    const uint32_t s_warp = (uint32_t)__cvta_generic_to_shared(wbase + (size_t)warp * pl.per_warp);
    const uint32_t s_hR = s_warp;                                 // [Rrows + 1][S][H]   (last row: trash)
    const uint32_t s_hP = s_hR + (uint32_t)S * (pl.nR + H) * 4u;  // [bins + 1][S][H]    (last row: trash)
    const uint32_t s_dsum = s_hP + (uint32_t)S * (pl.nP + H) * 4u;        // [H][pitch]
    const uint32_t s_cinfo = s_dsum + (uint32_t)(H * pl.pitch) * 4u;    // [pitch]: R row | P row << 16
    const uint32_t s_cdev = s_cinfo + (uint32_t)pl.pitch * 4u;    // [pitch]
    const uint32_t s_dlist = s_cdev + (uint32_t)pl.pitch * 4u;    // [pitch]: cells that need the slow path
    const uint32_t s_T = s_dlist + (uint32_t)pl.pitch * 4u;       // [H]
    const uint32_t s_hist = (ty ? s_hP : s_hR) + (uint32_t)(c2 * H + h) * 4u;       // + key * S * H * 4 B
    const uint32_t key_shift = ty ? 16u : 0u;
    const uint32_t trashR = (uint32_t)pl.Rrows, trashP = (uint32_t)num_bins;
    constexpr int hopw = HOPW;                                   // 32-bit words per walk (hops / 4)
    for (int i = threadIdx.x; i < (c.hops + 1) * 8; i += blockDim.x) XW[i] = (i & 7) < hopw ? expected_word(i >> 3, i & 7) : 0u;
    for (int i = threadIdx.x; i < 40; i += blockDim.x) invT[i] = 1.0f / (float)max(i, 1);
    for (int i = threadIdx.x; i < nwarp * pl.per_warp; i += blockDim.x) wbase[i] = 0.f;
    __syncthreads();
    const size_t hs = (size_t)c.T * c.Tp;
    const uint32_t pitch4 = (uint32_t)pl.pitch * 4u;
    float tacc = 0.f;
    for (int u = blockIdx.x * nwarp + warp; u < c.B * c.T; u += gridDim.x * nwarp) {
        const int g = u / c.T, a = u - g * c.T;
        const int n = c.n[g];
        if (a == 0 || a > n) continue;                       // row 0 carries no parameter (model_fqandtoyo.py:1160-1165)
        const int Tg = n + 1;
        const int64_t rowp = c.sq_off[g] + (int64_t)(a - 1) * n - 1;     // pair of cell b lives at rowp + b
        // ---- 1. sum phase: dsum[h][b] = sum over layers of plane[l][g][h][a][b]
        k2_bwd_sum_row<H>(dB + ((size_t)g * H * c.T + a) * c.Tp, Tg, nlayers, layer_stride, hs, s_dsum, pitch4, pl.pitch, lane);
        // ---- 2. index phase: cinfo[b] = R row | P row << 16 (the trash rows for cells that carry no gradient) ;
        //         cdev[b] = up to two deviating bytes ;  dlist = the cells that need the slow path
        int ndl = 0;
        const int Tg4 = (Tg + 3) & ~3;
        for (int bg = 0; bg < Tg4; bg += 32 * kIdxUnroll) {
          // the index bytes of up to kIdxUnroll x 32 cells are fetched before the first one is decoded: one memory latency per
          // group instead of one per 32 cells
          int rpv[kIdxUnroll], ppv[kIdxUnroll];
          uint32_t ewv[kIdxUnroll][HOPW];
#pragma unroll
          for (int u = 0; u < kIdxUnroll; ++u) {
              const int b = bg + 32 * u + lane;
              rpv[u] = ppv[u] = 0;
#pragma unroll
              for (int q = 0; q < HOPW; ++q) ewv[u][q] = 0u;
              if (b >= 1 && b < Tg) {
                  const int64_t pc = rowp + b;
                  rpv[u] = c.rel_pos[pc];
                  ppv[u] = c.poi_pos[pc];
                  const uint32_t *ei = reinterpret_cast<const uint32_t *>(c.edge_in + pc * c.hops);
#pragma unroll
                  for (int q = 0; q < HOPW; ++q) ewv[u][q] = __ldg(ei + q);
              }
          }
#pragma unroll
          for (int u = 0; u < kIdxUnroll; ++u) {
            const int b0 = bg + 32 * u;
            if (b0 >= Tg4) break;                                // warp-uniform
            const int b = b0 + lane;
            uint32_t info = trashR | (trashP << 16), dev = 0u, slow = 0u;
            if (b >= 1 && b < Tg) {
                const int rp = rpv[u], pp = ppv[u];
                const uint32_t(&ew)[HOPW] = ewv[u];
                const int rk = min(max(rp, 0), kRelRows - 1);
                const int L = expected_walk(rk, c.dk);
                const int row = (rk == 511) ? pl.Rrows - 1 : (rk < pl.Rrows - 1 ? rk : -1);
                if (rk - 1 < c.rel_pos_max) {                        // -inf entries carry no gradient
                    info = (row < 0 ? trashR : (uint32_t)row) | ((uint32_t)min(max(pp, 0), num_bins - 1) << 16);
                    int ndev = 0;
                    dev = (uint32_t)L << 2;
#pragma unroll
                    for (int q = 0; q < HOPW; ++q) {
                        uint32_t df = ew[q] ^ XW[L * 8 + q];
                        while (df != 0u) {
                            const int e = (__ffs(df) - 1) >> 3;
                            if (ndev < 2) dev |= (((uint32_t)(q * 4 + e) << 7) | ((ew[q] >> (8 * e)) & 0x7Fu)) << (8 + 12 * ndev);
                            ++ndev;
                            df &= ~(0xFFu << (8 * e));
                        }
                    }
                    dev |= (uint32_t)min(ndev, 3);
                    if (ndev || row < 0)
                        slow = (uint32_t)b | (row < 0 ? 1u << 12 : 0u) | (rk - 1 >= 510 ? 1u << 13 : 0u) | (ndev ? 1u << 14 : 0u) | (1u << 31);
                }
            }
            if (b < Tg4) {
                sts_u32(s_cinfo + (uint32_t)b * 4u, info);
                sts_u32(s_cdev + (uint32_t)b * 4u, dev);
            }
            const uint32_t bal = __ballot_sync(0xffffffffu, slow != 0u);
            if (slow) sts_u32(s_dlist + (uint32_t)(ndl + __popc(bal & ((1u << lane) - 1u))) * 4u, slow);
            ndl += __popc(bal);
          }
        }
        __syncwarp();
        // ---- 3. histogram phase: lane = (table, cell slot c2, head h)
        if (lane < H) tacc += lds_f32(s_dsum + (uint32_t)h * pitch4);          // column 0: graph-token virtual distance
        k2_bwd_hist_row<H>(s_cinfo, s_dsum, s_hist, key_shift, pitch4, Tg4, lane, c2, h);
        // ---- slow path (rare): walk bytes that differ from the expected walk, keys outside the plan; H lanes = H heads per
        //      listed cell, 32 / H cells at a time
        constexpr int SC = K2Heads<H>::kSlowCells;
        for (int e0 = 0; e0 < ndl; e0 += SC) {
            const int e = e0 + lane / H;
            if (e >= ndl || (SC * H < 32 && lane >= SC * H)) continue;
            const uint32_t ent = lds_u32(s_dlist + (uint32_t)e * 4u);
            const int b = ent & 0xFFF;
            const float d = lds_f32(s_dsum + (uint32_t)h * pitch4 + (uint32_t)b * 4u);
            if (ent & (1u << 12)) {
                // a key outside the plan has no histogram row, so the dRL unfold of the scatter kernel never sees it: its
                // expected-walk share d / sp for each of the L(rk) hops goes into dEW[k][dom] here (sp = L: rk >= 2 here)
                const int rk = min(max((int)c.rel_pos[rowp + b], 0), kRelRows - 1);
                fx_add(dR64 + rk * H + h, d);
                const int Lk = expected_walk(rk, c.dk);
                const float dl = d * invT[max(Lk, 1)];
                for (int k = 0; k < Lk; ++k) fx_add(sEW + (k * kSmallVocab + kDomEdge) * H + h, dl);
            }
            if (!(ent & (1u << 14))) continue;
            const uint32_t cd = lds_u32(s_cdev + (uint32_t)b * 4u);
            const int L = (cd >> 2) & 63, nd = cd & 3;
            const float dinv = d * invT[(ent & (1u << 13)) ? c.dk : max(L, 1)];
            if (nd <= 2) {
                for (int j = 0; j < nd; ++j) {
                    const uint32_t en = (cd >> (8 + 12 * j)) & 4095u;
                    const int k = en >> 7, v = en & 127, x = k < L ? kDomEdge : 0;
                    if (v != 0) {
                        if (v < kSmallVocab) fx_add(sEW + (k * kSmallVocab + v) * H + h, dinv);
                        else fx_add(dEWfull64 + ((size_t)k * kEdgeVocab + v) * H + h, dinv);
                    }
                    if (x != 0) fx_add(sEW + (k * kSmallVocab + x) * H + h, -dinv);
                }
            } else {
                const uint32_t *ei = reinterpret_cast<const uint32_t *>(c.edge_in + (rowp + b) * c.hops);
                for (int q = 0; q < hopw; ++q) {
                    const uint32_t ew = __ldg(ei + q), xw = XW[L * 8 + q];
                    uint32_t df = ew ^ xw;
                    while (df != 0u) {
                        const int eb = (__ffs(df) - 1) >> 3;
                        const int v = (ew >> (8 * eb)) & 0xFF, x = (xw >> (8 * eb)) & 0xFF;
                        const int k = q * 4 + eb;
                        if (v != 0) {
                            if (v < kSmallVocab) fx_add(sEW + (k * kSmallVocab + v) * H + h, dinv);
                            else fx_add(dEWfull64 + ((size_t)k * kEdgeVocab + min(v, kEdgeVocab - 1)) * H + h, dinv);
                        }
                        if (x != 0) fx_add(sEW + (k * kSmallVocab + x) * H + h, -dinv);
                        df &= ~(0xFFu << (8 * eb));
                    }
                }
            }
        }
        __syncwarp();
    }
    // column-0 sums: lanes 0..H-1 hold them
    if (lane < H) sts_f32(s_T + (uint32_t)h * 4u, tacc);
    __syncthreads();
    // CTA totals -> partial[blockIdx]
    float *out = partial + (size_t)blockIdx.x * pl.stride;
    for (int i = threadIdx.x; i < pl.nR; i += blockDim.x) {
        const int key = i / H, hh = i % H;
        float s = 0.f;
        for (int w = 0; w < nwarp; ++w)
            for (int r = 0; r < S; ++r) s += wbase[(size_t)w * pl.per_warp + (key * S + r) * H + hh];
        out[pl.nEWs + i] = s;
    }
    for (int i = threadIdx.x; i < pl.nP; i += blockDim.x) {
        const int key = i / H, hh = i % H;
        float s = 0.f;
        for (int w = 0; w < nwarp; ++w)
            for (int r = 0; r < S; ++r) s += wbase[(size_t)w * pl.per_warp + S * (pl.nR + H) + (key * S + r) * H + hh];
        out[pl.nEWs + pl.nR + i] = s;
    }
    if (threadIdx.x < H) {
        float s = 0.f;
        for (int w = 0; w < nwarp; ++w) s += wbase[(size_t)w * pl.per_warp + pl.per_warp - H + threadIdx.x];
        out[pl.nEWs + pl.nR + pl.nP + threadIdx.x] = s;
    }
}

// tot[i] = sum over CTAs of partial[cta][i] (fixed order); the EWsmall part [0, nEWs) is the exact integer sum of the CTAs'
// fixed-point tables.  The same launch converts the launch-wide fixed-point tables: dEWfull (threads [stride, stride + nEW))
// and the rel_pos overflow rows into dR (the next kRelRows * H threads).
template <int H>
__global__ void k2_bias_bwd_reduce_kernel(const float *__restrict__ partial, int nparts, int stride, int nEWs,
                                          const long long *__restrict__ ews64, float *__restrict__ tot,
                                          const long long *__restrict__ dEWfull64, int nEW, float *__restrict__ dEWfull,
                                          const long long *__restrict__ dR64, float *__restrict__ dR) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < nEWs) {
        long long s = 0;
#pragma unroll 8
        for (int p = 0; p < nparts; ++p) s += ews64[(size_t)p * nEWs + i];     // eight loads in flight; integer sum: any order
        tot[i] = fx_to_float(s);
    } else if (i < stride) {
        float s = 0.f;
#pragma unroll 8
        for (int p = 0; p < nparts; ++p) s += partial[(size_t)p * stride + i];  // loads hoisted, additions in part order
        tot[i] = s;
    } else if ((i -= stride) < nEW) {
        dEWfull[i] = fx_to_float(dEWfull64[i]);
    } else if ((i -= nEW) < kRelRows * H) {
        dR[i] = fx_to_float(dR64[i]);
    }
}

// totals -> dR, dPpos, dt, and the full dEW[k][v][h] (which already holds the global rare-path atomics):
//   dEW[k][v] += EWsmall[k][v] (v < 16) ;  dEW[k][dom] += sum_{rp : L(rp) > k} dRL[rp] / sp(rp)   (one warp per (k, h))
template <int H>
__global__ void k2_bias_bwd_scatter_kernel(const float *__restrict__ tot, const K2BwdPlan pl, int hops, int dk, int num_bins,
                                           float *__restrict__ dEWfull, float *__restrict__ dR, float *__restrict__ dP,
                                           float *__restrict__ dt) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const float *tE = tot, *tR = tot + pl.nEWs, *tP = tR + pl.nR, *tT = tP + pl.nP;
    if (i < kRelRows * H) {
        const int rp = i / H, hh = i % H;
        const int row = (rp == 511) ? pl.Rrows - 1 : (rp < pl.Rrows - 1 ? rp : -1);
        dR[i] += (row >= 0) ? tR[row * H + hh] : 0.f;     // dR holds the (normally empty) overflow atomics
    }
    if (i < num_bins * H) dP[i] = tP[i];
    if (i < H) dt[i] = tT[i];
    if (i < hops * kSmallVocab * H) {
        const int hh = i % H, v = (i / H) % kSmallVocab, k = i / (H * kSmallVocab);
        if (v != kDomEdge) dEWfull[((size_t)k * kEdgeVocab + v) * H + hh] += tE[i];
    }
    const int wid = i >> 5, lane = i & 31;
    if (wid < hops * H) {                                  // warp-uniform
        const int k = wid / H, hh = wid % H;
        float s = 0.f;
        for (int row = lane; row < pl.Rrows; row += 32) {
            const int rp = (row == pl.Rrows - 1) ? 511 : row;
            if (expected_walk(rp, dk) > k) s += tR[row * H + hh] / (float)min(max(rp - 1, 1), dk);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        if (lane == 0)
            dEWfull[((size_t)k * kEdgeVocab + kDomEdge) * H + hh] += s + tE[(k * kSmallVocab + kDomEdge) * H + hh];
    }
}

// dE[v][h'] = sum_k sum_h dEW[k][v][h] W[k][h'][h] ;  dW[k][h'][h] = sum_v E[v][h'] dEW[k][v][h]
template <int H>
__global__ void k2_bias_bwd_finish_kernel(const float *__restrict__ dEW, const float *__restrict__ E,
                                          const float *__restrict__ W, int hops, float *__restrict__ dE,
                                          float *__restrict__ dW) {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    const int nE = kEdgeVocab * H, nW = hops * H * H;
    if (idx < nE) {
        const int v = idx / H, hp = idx % H;
        float acc = 0.f;
        for (int k = 0; k < hops; ++k)
#pragma unroll
            for (int h = 0; h < H; ++h) acc += dEW[((size_t)k * kEdgeVocab + v) * H + h] * W[(k * H + hp) * H + h];
        dE[idx] = (v == 0) ? 0.f : acc;   // padding_idx row
    } else if (idx < nE + nW) {
        const int j = idx - nE;
        const int h = j % H, hp = (j / H) % H, k = j / (H * H);
        float acc = 0.f;
        for (int v = 0; v < kEdgeVocab; ++v) acc += E[v * H + hp] * dEW[((size_t)k * kEdgeVocab + v) * H + h];
        dW[j] = acc;
    }
}

// ---- direct edge encoding ----------------------------------------------------------------------------
// Graphormer's encoding for any edge_type other than multi_hop (the reference's else-branch between the multi-hop block,
// model_fqandtoyo.py:1168-1208, and the add into the bias, :1213-1216):
//   bias[g,h,a,b] = [a>=1, b>=1] ( R[rp[g,a-1,b-1],h] + Ppos[pp[g,a-1,b-1],h] + E[f[g,a-1,b-1],h] ) + [a>=1, b==0] t[h]
// with f = attn_edge_type (the packed u8 plane feat8: 0 for no edge, else count + 2) and -inf where rp-1 >= rel_pos_max.
// No walk, no edge_dis_encoder, no division by the distance.  E row 0 is read like any other row (cells without an edge).

// Forward.  Persistent CTAs; R (its -inf rows applied while staging), Ppos and E sit in shared memory.  Per cell 5 index bytes
// and three table gathers.  Cells per thread as in the multi-hop forward (K2FwdCells): at 8 heads a pair of adjacent cells
// (a, b) (a, b+1), b even; at 12 heads one cell (two cells keep 2 x 12 accumulators and three 12-float rows per cell live
// and spill 36-76 bytes per thread under __launch_bounds__(512, 2)).
template <int H, typename OutT>
__global__ void __launch_bounds__(512, 2) k2_direct_fwd_kernel(const K2Common c, const uint8_t *__restrict__ feat,
                                                               const float *__restrict__ Rg, const float *__restrict__ Pg,
                                                               int num_bins, const float *__restrict__ Eg,
                                                               const float *__restrict__ tvd, OutT *__restrict__ out) {
    extern __shared__ __align__(16) float sm[];
    const int nR = kRelRows * H, nP = num_bins * H, nE = kEdgeVocab * H;
    float *Rs = sm, *Ps = Rs + nR, *Es = Ps + nP;
    for (int i = threadIdx.x * 4; i < nR; i += blockDim.x * 4) {
        const float4 v = *reinterpret_cast<const float4 *>(Rg + i);
        *reinterpret_cast<float4 *>(Rs + i) = (i / H - 1 >= c.rel_pos_max) ? make_float4(-INFINITY, -INFINITY, -INFINITY, -INFINITY) : v;
    }
    for (int i = threadIdx.x * 4; i < nP; i += blockDim.x * 4)
        *reinterpret_cast<float4 *>(Ps + i) = *reinterpret_cast<const float4 *>(Pg + i);
    for (int i = threadIdx.x * 4; i < nE; i += blockDim.x * 4)
        *reinterpret_cast<float4 *>(Es + i) = *reinterpret_cast<const float4 *>(Eg + i);
    __syncthreads();
    constexpr int kCells = K2FwdCells<H>::kCells;
    const int half = c.Tp >> (kCells - 1);        // threads per plane row
    const int per_graph = c.T * half;
    const int tiles = ceil_div(per_graph, (int)blockDim.x);
    const uint64_t half_magic = ((1ull << 40) + half - 1) / half;     // f / half == (f * magic) >> 40 for f < 2^40 / half (> 2^30)
    const size_t hs = (size_t)c.T * c.Tp;
    for (int w = blockIdx.x; w < tiles * c.B; w += gridDim.x) {
        const int g = w / tiles, tile = w - g * tiles;
        const int n = c.n[g];
        const int Tg = n + 1;
        const int f = tile * blockDim.x + threadIdx.x;
        const int a = (int)(((uint64_t)f * half_magic) >> 40), b = (f - a * half) * kCells;
        if (a >= Tg || b >= Tg) continue;
        float acc[kCells][H];
#pragma unroll
        for (int s = 0; s < kCells; ++s)
#pragma unroll
            for (int h = 0; h < H; ++h) acc[s][h] = 0.f;
        if (a >= 1) {
            const int64_t rowp = c.sq_off[g] + (int64_t)(a - 1) * n;   // pair (a-1, j) lives at rowp + j
            // cell s of this thread is the pair j = b - 1 + s  (b == 0, s == 0: the virtual-distance column)
            int rp[kCells], pp[kCells], fe[kCells];
#pragma unroll
            for (int s = 0; s < kCells; ++s) {
                const int j = b - 1 + s;
                rp[s] = pp[s] = fe[s] = -1;
                if (j >= 0 && j < n) {
                    rp[s] = c.rel_pos[rowp + j];
                    pp[s] = c.poi_pos[rowp + j];
                    fe[s] = __ldg(feat + rowp + j);
                }
            }
#pragma unroll
            for (int s = 0; s < kCells; ++s) {
                if (fe[s] < 0) {
                    if (b == 0 && s == 0) {
#pragma unroll
                        for (int h = 0; h < H; ++h) acc[0][h] = __ldg(tvd + h);
                    }
                    continue;
                }
                float4 r0[H / 4], p0[H / 4], e0[H / 4];
                load_row<H>(r0, Rs + min(max(rp[s], 0), kRelRows - 1) * H);
                load_row<H>(p0, Ps + min(max(pp[s], 0), num_bins - 1) * H);
                load_row<H>(e0, Es + min(fe[s], kEdgeVocab - 1) * H);
#pragma unroll
                for (int i = 0; i < H / 4; ++i) {
                    acc[s][4 * i] = (r0[i].x + p0[i].x) + e0[i].x; acc[s][4 * i + 1] = (r0[i].y + p0[i].y) + e0[i].y;
                    acc[s][4 * i + 2] = (r0[i].z + p0[i].z) + e0[i].z; acc[s][4 * i + 3] = (r0[i].w + p0[i].w) + e0[i].w;
                }
            }
        }
        OutT *o = out + ((size_t)g * H * c.T + a) * c.Tp + b;
        if (kCells == 2 && b + 1 < Tg) {
#pragma unroll
            for (int h = 0; h < H; ++h) store2<OutT>(o + h * hs, acc[0][h], acc[kCells - 1][h]);
        } else {
#pragma unroll
            for (int h = 0; h < H; ++h) store1<OutT>(o + h * hs, acc[0][h]);
        }
    }
}

// Backward.  The multi-hop backward's row loop without the walk: per plane row (g, a) one warp runs the same sum phase and
// histogram phase (dR and dPpos as warp-private shared-memory histograms, dt from column 0).  The index phase packs only the
// R and P rows; cells with an edge (f != 0) and rel_pos keys outside the histogram plan go to a list that H lanes per cell
// work through: dE[f] by 64-bit fixed-point atomics into the CTA's [128][H] table in shared memory, out-of-plan keys into the
// launch-wide dR table in global memory.  Cells without an edge never touch dE: its row 0 (the padding row) stays 0.  On
// trajectory graphs a row has a few edges, so the list is short.  Integer sums do not depend on the order of the atomics, and
// the float histograms are reduced in a fixed order, so the result is bitwise reproducible.
template <int H>
static K2BwdPlan k2_direct_bwd_plan(int T, int num_bins) {
    constexpr int S = K2Heads<H>::kSlots;
    K2BwdPlan p = k2_bwd_plan<H>(T, round_up(T, 8), 0, num_bins);     // histogram rows and pitch as the multi-hop plan
    p.nEWs = 0;
    p.stride = p.nR + p.nP + H;                                         // partial row = [R | P | t(H)]
    p.per_warp = S * (p.nR + H) + S * (p.nP + H) + H * p.pitch + 2 * p.pitch + H;   // hR+trash | hP+trash | dsum | cinfo | dlist | t
    p.cta_words = 2 * kEdgeVocab * H;                                   // dE fixed-point table (long long)
    const int w = (int)((227 * 1024 - 2048 - p.cta_words * 4) / (p.per_warp * 4));
    p.warps = w > kK2BwdMaxWarps ? kK2BwdMaxWarps : w;
    return p;
}

// dlist entry: cell b (bits 0..11) | key outside the plan (bit 12) | edge (bit 13) | f (bits 14..20) | rel_pos key (bits 21..29)
constexpr uint32_t kDirOvf = 1u << 12, kDirEdge = 1u << 13;

template <int H, typename DT>
__global__ void __launch_bounds__(kK2BwdMaxWarps * 32, 1) k2_direct_bwd_kernel(const K2Common c, const uint8_t *__restrict__ feat,
                                                                               const DT *__restrict__ dB, int nlayers,
                                                                               int64_t layer_stride, int num_bins,
                                                                               const K2BwdPlan pl, float *__restrict__ partial,
                                                                               long long *__restrict__ dE64,
                                                                               long long *__restrict__ dR64) {
    extern __shared__ __align__(16) float sm[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = blockDim.x >> 5;
    constexpr int S = K2Heads<H>::kSlots;
    const int ty = lane / (S * H), c2 = (lane / H) % S, h = lane % H;      // table (0 = R, 1 = P), cell slot, head
    long long *sE = reinterpret_cast<long long *>(sm);            // [128][H] fixed point
    float *wbase = sm + pl.cta_words;
    const uint32_t s_warp = (uint32_t)__cvta_generic_to_shared(wbase + (size_t)warp * pl.per_warp);
    const uint32_t s_hR = s_warp;                                 // [Rrows + 1][S][H]   (last row: trash)
    const uint32_t s_hP = s_hR + (uint32_t)S * (pl.nR + H) * 4u;  // [bins + 1][S][H]    (last row: trash)
    const uint32_t s_dsum = s_hP + (uint32_t)S * (pl.nP + H) * 4u;        // [H][pitch]
    const uint32_t s_cinfo = s_dsum + (uint32_t)(H * pl.pitch) * 4u;    // [pitch]: R row | P row << 16
    const uint32_t s_dlist = s_cinfo + (uint32_t)pl.pitch * 4u;   // [pitch]: cells for the list path
    const uint32_t s_T = s_dlist + (uint32_t)pl.pitch * 4u;       // [H]
    const uint32_t s_hist = (ty ? s_hP : s_hR) + (uint32_t)(c2 * H + h) * 4u;
    const uint32_t key_shift = ty ? 16u : 0u;
    const uint32_t trashR = (uint32_t)pl.Rrows, trashP = (uint32_t)num_bins;
    for (int i = threadIdx.x; i < kEdgeVocab * H; i += blockDim.x) sE[i] = 0;
    for (int i = threadIdx.x; i < nwarp * pl.per_warp; i += blockDim.x) wbase[i] = 0.f;
    __syncthreads();
    const size_t hs = (size_t)c.T * c.Tp;
    const uint32_t pitch4 = (uint32_t)pl.pitch * 4u;
    float tacc = 0.f;
    for (int u = blockIdx.x * nwarp + warp; u < c.B * c.T; u += gridDim.x * nwarp) {
        const int g = u / c.T, a = u - g * c.T;
        const int n = c.n[g];
        if (a == 0 || a > n) continue;                       // row 0 carries no parameter (model_fqandtoyo.py:1160-1165)
        const int Tg = n + 1;
        const int64_t rowp = c.sq_off[g] + (int64_t)(a - 1) * n - 1;     // pair of cell b lives at rowp + b
        // ---- 1. sum phase
        k2_bwd_sum_row<H>(dB + ((size_t)g * H * c.T + a) * c.Tp, Tg, nlayers, layer_stride, hs, s_dsum, pitch4, pl.pitch, lane);
        // ---- 2. index phase: cinfo[b] = R row | P row << 16 (the trash rows for cells that carry no gradient); dlist
        int ndl = 0;
        const int Tg4 = (Tg + 3) & ~3;
        for (int bg = 0; bg < Tg4; bg += 32 * kIdxUnroll) {
            int rpv[kIdxUnroll], ppv[kIdxUnroll], fv[kIdxUnroll];
#pragma unroll
            for (int u2 = 0; u2 < kIdxUnroll; ++u2) {
                const int b = bg + 32 * u2 + lane;
                rpv[u2] = ppv[u2] = fv[u2] = 0;
                if (b >= 1 && b < Tg) {
                    rpv[u2] = c.rel_pos[rowp + b];
                    ppv[u2] = c.poi_pos[rowp + b];
                    fv[u2] = __ldg(feat + rowp + b);
                }
            }
#pragma unroll
            for (int u2 = 0; u2 < kIdxUnroll; ++u2) {
                const int b0 = bg + 32 * u2;
                if (b0 >= Tg4) break;                            // warp-uniform
                const int b = b0 + lane;
                uint32_t info = trashR | (trashP << 16), ent = 0u;
                if (b >= 1 && b < Tg) {
                    const int rk = min(max(rpv[u2], 0), kRelRows - 1);
                    const int row = (rk == 511) ? pl.Rrows - 1 : (rk < pl.Rrows - 1 ? rk : -1);
                    if (rk - 1 < c.rel_pos_max) {                    // -inf entries carry no gradient
                        info = (row < 0 ? trashR : (uint32_t)row) | ((uint32_t)min(max(ppv[u2], 0), num_bins - 1) << 16);
                        const uint32_t fe = (uint32_t)min(fv[u2], kEdgeVocab - 1);
                        if (fe != 0u || row < 0)
                            ent = (uint32_t)b | (row < 0 ? kDirOvf : 0u) | (fe != 0u ? kDirEdge : 0u) | (fe << 14) | ((uint32_t)rk << 21);
                    }
                }
                if (b < Tg4) sts_u32(s_cinfo + (uint32_t)b * 4u, info);
                const uint32_t bal = __ballot_sync(0xffffffffu, ent != 0u);
                if (ent) sts_u32(s_dlist + (uint32_t)(ndl + __popc(bal & ((1u << lane) - 1u))) * 4u, ent);
                ndl += __popc(bal);
            }
        }
        __syncwarp();
        // ---- 3. histogram phase
        if (lane < H) tacc += lds_f32(s_dsum + (uint32_t)h * pitch4);          // column 0: graph-token virtual distance
        k2_bwd_hist_row<H>(s_cinfo, s_dsum, s_hist, key_shift, pitch4, Tg4, lane, c2, h);
        // ---- list path: H lanes = H heads per listed cell, 32 / H cells at a time
        constexpr int SC = K2Heads<H>::kSlowCells;
        for (int e0 = 0; e0 < ndl; e0 += SC) {
            const int e = e0 + lane / H;
            if (e >= ndl || (SC * H < 32 && lane >= SC * H)) continue;
            const uint32_t ent = lds_u32(s_dlist + (uint32_t)e * 4u);
            const float d = lds_f32(s_dsum + (uint32_t)h * pitch4 + (ent & 0xFFFu) * 4u);
            if (ent & kDirOvf) fx_add(dR64 + (ent >> 21) * H + h, d);
            if (ent & kDirEdge) fx_add(sE + ((ent >> 14) & 127u) * H + h, d);
        }
        __syncwarp();
    }
    if (lane < H) sts_f32(s_T + (uint32_t)h * 4u, tacc);
    __syncthreads();
    // CTA totals: histograms -> partial[blockIdx] (summed in a fixed order later), dE table -> the launch-wide one
    float *out = partial + (size_t)blockIdx.x * pl.stride;
    for (int i = threadIdx.x; i < pl.nR; i += blockDim.x) {
        const int key = i / H, hh = i % H;
        float s = 0.f;
        for (int w = 0; w < nwarp; ++w)
            for (int r = 0; r < S; ++r) s += wbase[(size_t)w * pl.per_warp + (key * S + r) * H + hh];
        out[i] = s;
    }
    for (int i = threadIdx.x; i < pl.nP; i += blockDim.x) {
        const int key = i / H, hh = i % H;
        float s = 0.f;
        for (int w = 0; w < nwarp; ++w)
            for (int r = 0; r < S; ++r) s += wbase[(size_t)w * pl.per_warp + S * (pl.nR + H) + (key * S + r) * H + hh];
        out[pl.nR + i] = s;
    }
    if (threadIdx.x < H) {
        float s = 0.f;
        for (int w = 0; w < nwarp; ++w) s += wbase[(size_t)w * pl.per_warp + pl.per_warp - H + threadIdx.x];
        out[pl.nR + pl.nP + threadIdx.x] = s;
    }
    for (int i = threadIdx.x; i < kEdgeVocab * H; i += blockDim.x)
        if (sE[i] != 0) atomicAdd(reinterpret_cast<unsigned long long *>(dE64 + i), (unsigned long long)sE[i]);
}

}  // namespace mobgt

using namespace mobgt;

// head counts the kernels are instantiated for (K2Heads); any other value is MOBGT_ERR_UNSUPPORTED
static bool k2_heads_built(int H) { return H == 8 || H == 12; }

extern "C" int64_t mobgt_bias_fwd_workspace_bytes(int32_t hops, int32_t H) {
    if (!k2_heads_built(H) || hops < 4 || hops > MOBGT_MAX_HOPS || hops % 4 != 0) return -1;
    return (int64_t)(hops * kEdgeVocab + kRelRows) * H * (int64_t)sizeof(float);
}

template <int H>
static int32_t bias_fwd(const int32_t *n, const int64_t *sq_off, const int16_t *rel_pos, const int16_t *poi_pos,
                        const uint8_t *edge_in, int32_t B, int32_t T, int32_t Tp, int32_t hops, int32_t dk, int32_t rel_pos_max,
                        int32_t num_bins, const float *R, const float *Ppos, const float *E, const float *W, const float *tvd,
                        void *workspace, void *out, int32_t out_dtype, cudaStream_t s) {
    float *EW = static_cast<float *>(workspace);                 // [hops][128][H] then RL [512][H]
    const int tabn = hops * kEdgeVocab * H;
    float *RL = EW + tabn;
    k2_prep_kernel<H><<<ceil_div(tabn + kRelRows * H, 256), 256, 0, s>>>(E, W, R, hops, dk, rel_pos_max, EW, RL);
    MOBGT_LAUNCH_OK("k2_prep_kernel");
    K2Common c{n, sq_off, rel_pos, poi_pos, edge_in, B, T, Tp, hops, rel_pos_max, dk};
    const size_t smem = (size_t)(kRelRows * H + num_bins * H + (hops + 1) * 8) * sizeof(float);
    const int tiles_total = ceil_div(T * (Tp / K2FwdCells<H>::kCells), 512) * B;
    dim3 grid((unsigned)min(2 * kNumSMs, tiles_total));
    auto launch = [&](auto kern, auto *o) -> int32_t {
        MOBGT_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        kern<<<grid, 512, smem, s>>>(c, RL, Ppos, num_bins, tvd, EW, o);
        return MOBGT_OK;
    };
    int32_t rc = MOBGT_OK;
#define MOBGT_K2_CASE(HW)                                                                                                \
    case HW:                                                                                                             \
        rc = (out_dtype == MOBGT_F32) ? launch(k2_bias_fwd_kernel<H, float, HW>, static_cast<float *>(out))              \
                                      : launch(k2_bias_fwd_kernel<H, __nv_bfloat16, HW>, static_cast<__nv_bfloat16 *>(out)); \
        break;
    switch (hops / 4) {
        MOBGT_K2_CASE(1) MOBGT_K2_CASE(2) MOBGT_K2_CASE(3) MOBGT_K2_CASE(4) MOBGT_K2_CASE(5) MOBGT_K2_CASE(6) MOBGT_K2_CASE(7)
        MOBGT_K2_CASE(8)
        default: MOBGT_REQUIRE(false, MOBGT_ERR_BAD_SHAPE, "mobgt_bias_fwd: hops=%d", hops);
    }
#undef MOBGT_K2_CASE
    if (rc) return rc;
    MOBGT_LAUNCH_OK("k2_bias_fwd_kernel");
    return MOBGT_OK;
}

extern "C" int32_t mobgt_bias_fwd(const int32_t *n, const int64_t *sq_off, const int16_t *rel_pos, const int16_t *poi_pos,
                                  const uint8_t *edge_in, int32_t B, int32_t T, int32_t Tp, int32_t hops, int32_t dk, int32_t H,
                                  int32_t rel_pos_max, int32_t num_bins, const float *R, const float *Ppos, const float *E,
                                  const float *W, const float *tvd, void *workspace, void *out, int32_t out_dtype,
                                  void *stream) {
    MOBGT_REQUIRE(k2_heads_built(H), MOBGT_ERR_UNSUPPORTED, "mobgt_bias_fwd: num_heads=%d is not built (8 and 12 heads)", H);
    MOBGT_REQUIRE(n && sq_off && rel_pos && poi_pos && edge_in && R && Ppos && E && W && tvd && workspace && out,
                  MOBGT_ERR_NULL, "mobgt_bias_fwd: null pointer");
    MOBGT_REQUIRE(hops >= 4 && hops <= MOBGT_MAX_HOPS && hops % 4 == 0, MOBGT_ERR_BAD_SHAPE,
                  "mobgt_bias_fwd: hops=%d must be a multiple of 4 in [4,%d]", hops, MOBGT_MAX_HOPS);
    MOBGT_REQUIRE(dk >= 1 && dk <= hops, MOBGT_ERR_BAD_SHAPE, "mobgt_bias_fwd: dk=%d outside [1, hops=%d]", dk, hops);
    MOBGT_REQUIRE(num_bins >= 1 && num_bins <= 1024, MOBGT_ERR_BAD_SHAPE, "mobgt_bias_fwd: num_bins=%d", num_bins);
    MOBGT_REQUIRE(T >= 2 && T <= MOBGT_MAX_MODEL_NODES + 1 && Tp >= T && Tp % 8 == 0, MOBGT_ERR_BAD_SHAPE,
                  "mobgt_bias_fwd: T=%d Tp=%d (T <= 1025: graphs of at most 1024 nodes)", T, Tp);
    MOBGT_REQUIRE(out_dtype == MOBGT_F32 || out_dtype == MOBGT_BF16, MOBGT_ERR_BAD_DTYPE, "mobgt_bias_fwd: dtype");
    if (B <= 0) return MOBGT_OK;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    auto f = H == 8 ? bias_fwd<8> : bias_fwd<12>;
    return f(n, sq_off, rel_pos, poi_pos, edge_in, B, T, Tp, hops, dk, rel_pos_max, num_bins, R, Ppos, E, W, tvd, workspace, out,
             out_dtype, s);
}

// 64-bit words of the fixed-point rare-path tables: per-CTA EWsmall | launch-wide dEW | rel_pos overflow rows
template <int H>
static int64_t k2_bwd_fx_words(int hops, const K2BwdPlan &pl) {
    return (int64_t)kNumSMs * pl.nEWs + (int64_t)hops * kEdgeVocab * H + (int64_t)kRelRows * H;
}

template <int H>
static int64_t bias_bwd_workspace_bytes(int32_t T, int32_t hops, int32_t num_bins) {
    if (T < 2 || hops < 4 || hops > MOBGT_MAX_HOPS || num_bins < 1 || num_bins > 1024) return -1;
    const K2BwdPlan pl = k2_bwd_plan<H>(T, round_up(T, 8), hops, num_bins);
    return ((int64_t)hops * kEdgeVocab * H + (int64_t)(kNumSMs + 1) * pl.stride) * (int64_t)sizeof(float) + 16 +
           k2_bwd_fx_words<H>(hops, pl) * (int64_t)sizeof(long long);
}

extern "C" int64_t mobgt_bias_bwd_workspace_bytes(int32_t T, int32_t hops, int32_t num_bins) {
    return bias_bwd_workspace_bytes<8>(T, hops, num_bins);
}

extern "C" int64_t mobgt_bias_bwd_heads_workspace_bytes(int32_t T, int32_t hops, int32_t num_bins, int32_t H) {
    if (!k2_heads_built(H)) return -1;
    return H == 8 ? bias_bwd_workspace_bytes<8>(T, hops, num_bins) : bias_bwd_workspace_bytes<12>(T, hops, num_bins);
}

template <int H>
static int32_t bias_bwd(const int32_t *n, const int64_t *sq_off, const int16_t *rel_pos, const int16_t *poi_pos,
                        const uint8_t *edge_in, int32_t B, int32_t T, int32_t Tp, int32_t hops, int32_t dk, int32_t rel_pos_max,
                        int32_t num_bins, const void *dBias, int32_t dbias_dtype, int32_t n_layers, int64_t layer_stride,
                        const float *E, const float *W, void *workspace, int64_t workspace_bytes, float *dR, float *dPpos,
                        float *dE, float *dW, float *dtvd, cudaStream_t s) {
    const K2BwdPlan pl = k2_bwd_plan<H>(T, Tp, hops, num_bins);
    MOBGT_REQUIRE(pl.warps >= 1, MOBGT_ERR_UNSUPPORTED, "mobgt_bias_bwd: no shared-memory plan for T=%d bins=%d", T, num_bins);
    const int64_t nEW = (int64_t)hops * kEdgeVocab * H;
    const int64_t nfloat = nEW + (int64_t)(kNumSMs + 1) * pl.stride;
    const int64_t fx_off = (nfloat * (int64_t)sizeof(float) + 15) / 16 * 16;
    const int64_t need = fx_off + k2_bwd_fx_words<H>(hops, pl) * (int64_t)sizeof(long long);
    MOBGT_REQUIRE(workspace_bytes >= need, MOBGT_ERR_WORKSPACE_TOO_SMALL, "mobgt_bias_bwd: workspace %lld < %lld bytes",
                  (long long)workspace_bytes, (long long)need);
    float *dEWfull = static_cast<float *>(workspace);      // [hops][128][H], then [stride] totals, then [kNumSMs][stride] partials
    float *tot = dEWfull + nEW;
    float *partial = tot + pl.stride;
    MOBGT_REQUIRE(((uintptr_t)workspace & 15) == 0, MOBGT_ERR_BAD_SHAPE, "mobgt_bias_bwd: workspace must be 16-byte aligned");
    long long *ews64 = reinterpret_cast<long long *>(static_cast<char *>(workspace) + fx_off);   // [kNumSMs][nEWs]
    long long *dEWfull64 = ews64 + (size_t)kNumSMs * pl.nEWs;                                     // [hops][128][H]
    long long *dR64 = dEWfull64 + nEW;                                                            // [512][H]
    MOBGT_CUDA_OK(cudaMemsetAsync(ews64, 0, (size_t)k2_bwd_fx_words<H>(hops, pl) * sizeof(long long), s));
    const int nparts = B > 0 ? kNumSMs : 0;
    if (B > 0) {
        K2Common c{n, sq_off, rel_pos, poi_pos, edge_in, B, T, Tp, hops, rel_pos_max, dk};
        const size_t smem = (size_t)(pl.cta_words + pl.warps * pl.per_warp) * sizeof(float);
        auto launch = [&](auto kern, auto *db, int nl, int64_t ls) -> int32_t {
            MOBGT_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            kern<<<kNumSMs, pl.warps * 32, smem, s>>>(c, db, nl, ls, num_bins, pl, partial, ews64, dEWfull64, dR64);
            return MOBGT_OK;
        };
        int32_t rc = MOBGT_OK;
#define MOBGT_K2B_CASE(HW)                                                                                                   \
    case HW:                                                                                                                 \
        rc = (dbias_dtype == MOBGT_F32)                                                                                      \
                 ? launch(k2_bias_bwd_kernel<H, float, HW>, static_cast<const float *>(dBias), 1, (int64_t)0)                \
                 : launch(k2_bias_bwd_kernel<H, __nv_bfloat16, HW>, static_cast<const __nv_bfloat16 *>(dBias), n_layers,     \
                          layer_stride);                                                                                     \
        break;
        switch (hops / 4) {
            MOBGT_K2B_CASE(1) MOBGT_K2B_CASE(2) MOBGT_K2B_CASE(3) MOBGT_K2B_CASE(4) MOBGT_K2B_CASE(5) MOBGT_K2B_CASE(6)
            MOBGT_K2B_CASE(7) MOBGT_K2B_CASE(8)
            default: MOBGT_REQUIRE(false, MOBGT_ERR_BAD_SHAPE, "mobgt_bias_bwd: hops=%d", hops);
        }
#undef MOBGT_K2B_CASE
        if (rc) return rc;
        MOBGT_LAUNCH_OK("k2_bias_bwd_kernel");
    }
    k2_bias_bwd_reduce_kernel<H><<<ceil_div(pl.stride + (int)nEW + kRelRows * H, 256), 256, 0, s>>>(
        partial, nparts, pl.stride, pl.nEWs, ews64, tot, dEWfull64, (int)nEW, dEWfull, dR64, dR);
    MOBGT_LAUNCH_OK("k2_bias_bwd_reduce_kernel");
    k2_bias_bwd_scatter_kernel<H><<<ceil_div(max(max(kRelRows, num_bins) * H, hops * H * 32), 256), 256, 0, s>>>(
        tot, pl, hops, dk, num_bins, dEWfull, dR, dPpos, dtvd);
    MOBGT_LAUNCH_OK("k2_bias_bwd_scatter_kernel");
    k2_bias_bwd_finish_kernel<H><<<ceil_div(kEdgeVocab * H + hops * H * H, 256), 256, 0, s>>>(dEWfull, E, W, hops, dE, dW);
    MOBGT_LAUNCH_OK("k2_bias_bwd_finish_kernel");
    return MOBGT_OK;
}

extern "C" int32_t mobgt_bias_bwd(const int32_t *n, const int64_t *sq_off, const int16_t *rel_pos, const int16_t *poi_pos,
                                  const uint8_t *edge_in, int32_t B, int32_t T, int32_t Tp, int32_t hops, int32_t dk, int32_t H,
                                  int32_t rel_pos_max, int32_t num_bins, const void *dBias, int32_t dbias_dtype,
                                  int32_t n_layers, int64_t layer_stride, const float *E, const float *W,
                                  void *workspace, int64_t workspace_bytes, float *dR, float *dPpos, float *dE, float *dW,
                                  float *dtvd, void *stream) {
    MOBGT_REQUIRE(k2_heads_built(H), MOBGT_ERR_UNSUPPORTED, "mobgt_bias_bwd: num_heads=%d is not built (8 and 12 heads)", H);
    MOBGT_REQUIRE(n && sq_off && rel_pos && poi_pos && edge_in && dBias && E && W && workspace && dR && dPpos && dE && dW && dtvd,
                  MOBGT_ERR_NULL, "mobgt_bias_bwd: null pointer");
    MOBGT_REQUIRE(hops >= 4 && hops <= MOBGT_MAX_HOPS && hops % 4 == 0 && num_bins >= 1 && num_bins <= 1024, MOBGT_ERR_BAD_SHAPE,
                  "mobgt_bias_bwd: hops=%d num_bins=%d", hops, num_bins);
    MOBGT_REQUIRE(dk >= 1 && dk <= hops, MOBGT_ERR_BAD_SHAPE, "mobgt_bias_bwd: dk=%d outside [1, hops=%d]", dk, hops);
    MOBGT_REQUIRE(T >= 2 && T <= MOBGT_MAX_MODEL_NODES + 1 && Tp >= T && Tp % 8 == 0, MOBGT_ERR_BAD_SHAPE,
                  "mobgt_bias_bwd: T=%d Tp=%d (T <= 1025: graphs of at most 1024 nodes)", T, Tp);
    MOBGT_REQUIRE((dbias_dtype == MOBGT_F32 && n_layers == 1) || (dbias_dtype == MOBGT_BF16 && n_layers >= 1 && n_layers <= 64),
                  MOBGT_ERR_BAD_DTYPE, "mobgt_bias_bwd: dbias dtype %d with %d layer planes", dbias_dtype, n_layers);
    MOBGT_REQUIRE(((uintptr_t)dBias & 15) == 0 && (dbias_dtype == MOBGT_F32 || layer_stride % 8 == 0), MOBGT_ERR_BAD_SHAPE,
                  "mobgt_bias_bwd: dBias planes must be 16-byte aligned");
    auto f = H == 8 ? bias_bwd<8> : bias_bwd<12>;
    return f(n, sq_off, rel_pos, poi_pos, edge_in, B, T, Tp, hops, dk, rel_pos_max, num_bins, dBias, dbias_dtype, n_layers,
             layer_stride, E, W, workspace, workspace_bytes, dR, dPpos, dE, dW, dtvd, static_cast<cudaStream_t>(stream));
}

// ---- direct edge encoding: entry points ----

template <int H>
static int32_t bias_direct_fwd(const K2Common &c, const uint8_t *feat, int32_t num_bins, const float *R, const float *Ppos,
                               const float *E, const float *tvd, void *out, int32_t out_dtype, cudaStream_t s) {
    const size_t smem = (size_t)(kRelRows + num_bins + kEdgeVocab) * H * sizeof(float);
    const int tiles_total = ceil_div(c.T * (c.Tp / K2FwdCells<H>::kCells), 512) * c.B;
    dim3 grid((unsigned)min(2 * kNumSMs, tiles_total));
    auto launch = [&](auto kern, auto *o) -> int32_t {
        MOBGT_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        kern<<<grid, 512, smem, s>>>(c, feat, R, Ppos, num_bins, E, tvd, o);
        return MOBGT_OK;
    };
    const int32_t rc = (out_dtype == MOBGT_F32) ? launch(k2_direct_fwd_kernel<H, float>, static_cast<float *>(out))
                                                : launch(k2_direct_fwd_kernel<H, __nv_bfloat16>, static_cast<__nv_bfloat16 *>(out));
    if (rc) return rc;
    MOBGT_LAUNCH_OK("k2_direct_fwd_kernel");
    return MOBGT_OK;
}

extern "C" int32_t mobgt_bias_direct_fwd(const int32_t *n, const int64_t *sq_off, const int16_t *rel_pos, const int16_t *poi_pos,
                                         const uint8_t *feat, int32_t B, int32_t T, int32_t Tp, int32_t H, int32_t rel_pos_max,
                                         int32_t num_bins, const float *R, const float *Ppos, const float *E, const float *tvd,
                                         void *out, int32_t out_dtype, void *stream) {
    MOBGT_REQUIRE(k2_heads_built(H), MOBGT_ERR_UNSUPPORTED, "mobgt_bias_direct_fwd: num_heads=%d is not built (8 and 12 heads)", H);
    MOBGT_REQUIRE(n && sq_off && rel_pos && poi_pos && feat && R && Ppos && E && tvd && out, MOBGT_ERR_NULL,
                  "mobgt_bias_direct_fwd: null pointer");
    MOBGT_REQUIRE(num_bins >= 1 && num_bins <= 1024, MOBGT_ERR_BAD_SHAPE, "mobgt_bias_direct_fwd: num_bins=%d", num_bins);
    MOBGT_REQUIRE(T >= 2 && T <= MOBGT_MAX_MODEL_NODES + 1 && Tp >= T && Tp % 8 == 0, MOBGT_ERR_BAD_SHAPE,
                  "mobgt_bias_direct_fwd: T=%d Tp=%d (T <= 1025: graphs of at most 1024 nodes)", T, Tp);
    MOBGT_REQUIRE(out_dtype == MOBGT_F32 || out_dtype == MOBGT_BF16, MOBGT_ERR_BAD_DTYPE, "mobgt_bias_direct_fwd: dtype");
    if (B <= 0) return MOBGT_OK;
    const K2Common c{n, sq_off, rel_pos, poi_pos, nullptr, B, T, Tp, 0, rel_pos_max, 0};
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    auto f = H == 8 ? bias_direct_fwd<8> : bias_direct_fwd<12>;
    return f(c, feat, num_bins, R, Ppos, E, tvd, out, out_dtype, s);
}

// workspace of the direct backward: [stride] totals, [kNumSMs][stride] partials, then (16-byte aligned) the fixed-point dE
// [128][H] and rel_pos overflow [512][H] tables
template <int H>
static int64_t direct_fx_offset(const K2BwdPlan &pl) {
    return ((int64_t)(kNumSMs + 1) * pl.stride * (int64_t)sizeof(float) + 15) / 16 * 16;
}
template <int H>
static int64_t direct_bwd_workspace_bytes(int32_t T, int32_t num_bins) {
    const K2BwdPlan pl = k2_direct_bwd_plan<H>(T, num_bins);
    return direct_fx_offset<H>(pl) + (int64_t)(kEdgeVocab + kRelRows) * H * (int64_t)sizeof(long long);
}

extern "C" int64_t mobgt_bias_direct_bwd_workspace_bytes(int32_t T, int32_t num_bins, int32_t H) {
    if (!k2_heads_built(H) || T < 2 || num_bins < 1 || num_bins > 1024) return -1;
    return H == 8 ? direct_bwd_workspace_bytes<8>(T, num_bins) : direct_bwd_workspace_bytes<12>(T, num_bins);
}

template <int H>
static int32_t bias_direct_bwd(const K2Common &c, const uint8_t *feat, int32_t num_bins, const void *dBias, int32_t dbias_dtype,
                               int32_t n_layers, int64_t layer_stride, void *workspace, int64_t workspace_bytes, float *dR,
                               float *dPpos, float *dE, float *dtvd, cudaStream_t s) {
    const K2BwdPlan pl = k2_direct_bwd_plan<H>(c.T, num_bins);
    MOBGT_REQUIRE(pl.warps >= 1, MOBGT_ERR_UNSUPPORTED, "mobgt_bias_direct_bwd: no shared-memory plan for T=%d bins=%d", c.T,
                  num_bins);
    const int64_t fx_off = direct_fx_offset<H>(pl);
    const int64_t need = direct_bwd_workspace_bytes<H>(c.T, num_bins);
    MOBGT_REQUIRE(workspace_bytes >= need, MOBGT_ERR_WORKSPACE_TOO_SMALL, "mobgt_bias_direct_bwd: workspace %lld < %lld bytes",
                  (long long)workspace_bytes, (long long)need);
    MOBGT_REQUIRE(((uintptr_t)workspace & 15) == 0, MOBGT_ERR_BAD_SHAPE, "mobgt_bias_direct_bwd: workspace must be 16-byte aligned");
    float *tot = static_cast<float *>(workspace);          // [stride] totals, then [kNumSMs][stride] partials
    float *partial = tot + pl.stride;
    long long *dE64 = reinterpret_cast<long long *>(static_cast<char *>(workspace) + fx_off);   // [128][H]
    long long *dR64 = dE64 + kEdgeVocab * H;                                                     // [512][H]
    MOBGT_CUDA_OK(cudaMemsetAsync(dE64, 0, (size_t)(kEdgeVocab + kRelRows) * H * sizeof(long long), s));
    const int nparts = c.B > 0 ? kNumSMs : 0;
    if (c.B > 0) {
        const size_t smem = (size_t)(pl.cta_words + pl.warps * pl.per_warp) * sizeof(float);
        auto launch = [&](auto kern, auto *db, int nl, int64_t ls) -> int32_t {
            MOBGT_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            kern<<<kNumSMs, pl.warps * 32, smem, s>>>(c, feat, db, nl, ls, num_bins, pl, partial, dE64, dR64);
            return MOBGT_OK;
        };
        const int32_t rc = (dbias_dtype == MOBGT_F32)
                               ? launch(k2_direct_bwd_kernel<H, float>, static_cast<const float *>(dBias), 1, (int64_t)0)
                               : launch(k2_direct_bwd_kernel<H, __nv_bfloat16>, static_cast<const __nv_bfloat16 *>(dBias),
                                        n_layers, layer_stride);
        if (rc) return rc;
        MOBGT_LAUNCH_OK("k2_direct_bwd_kernel");
    }
    // the multi-hop epilogue without its walk tables: fixed-order partial sums, the fixed-point dE and overflow rows to fp32,
    // then the histogram rows into dR / dPpos / dt
    k2_bias_bwd_reduce_kernel<H><<<ceil_div(pl.stride + (kEdgeVocab + kRelRows) * H, 256), 256, 0, s>>>(
        partial, nparts, pl.stride, 0, nullptr, tot, dE64, kEdgeVocab * H, dE, dR64, dR);
    MOBGT_LAUNCH_OK("k2_bias_bwd_reduce_kernel");
    k2_bias_bwd_scatter_kernel<H><<<ceil_div(max(kRelRows, num_bins) * H, 256), 256, 0, s>>>(tot, pl, 0, 1, num_bins, nullptr, dR,
                                                                                            dPpos, dtvd);
    MOBGT_LAUNCH_OK("k2_bias_bwd_scatter_kernel");
    return MOBGT_OK;
}

extern "C" int32_t mobgt_bias_direct_bwd(const int32_t *n, const int64_t *sq_off, const int16_t *rel_pos, const int16_t *poi_pos,
                                         const uint8_t *feat, int32_t B, int32_t T, int32_t Tp, int32_t H, int32_t rel_pos_max,
                                         int32_t num_bins, const void *dBias, int32_t dbias_dtype, int32_t n_layers,
                                         int64_t layer_stride, void *workspace, int64_t workspace_bytes, float *dR, float *dPpos,
                                         float *dE, float *dtvd, void *stream) {
    MOBGT_REQUIRE(k2_heads_built(H), MOBGT_ERR_UNSUPPORTED, "mobgt_bias_direct_bwd: num_heads=%d is not built (8 and 12 heads)", H);
    MOBGT_REQUIRE(n && sq_off && rel_pos && poi_pos && feat && dBias && workspace && dR && dPpos && dE && dtvd, MOBGT_ERR_NULL,
                  "mobgt_bias_direct_bwd: null pointer");
    MOBGT_REQUIRE(num_bins >= 1 && num_bins <= 1024, MOBGT_ERR_BAD_SHAPE, "mobgt_bias_direct_bwd: num_bins=%d", num_bins);
    MOBGT_REQUIRE(T >= 2 && T <= MOBGT_MAX_MODEL_NODES + 1 && Tp >= T && Tp % 8 == 0, MOBGT_ERR_BAD_SHAPE,
                  "mobgt_bias_direct_bwd: T=%d Tp=%d (T <= 1025: graphs of at most 1024 nodes)", T, Tp);
    MOBGT_REQUIRE((dbias_dtype == MOBGT_F32 && n_layers == 1) || (dbias_dtype == MOBGT_BF16 && n_layers >= 1 && n_layers <= 64),
                  MOBGT_ERR_BAD_DTYPE, "mobgt_bias_direct_bwd: dbias dtype %d with %d layer planes", dbias_dtype, n_layers);
    MOBGT_REQUIRE(((uintptr_t)dBias & 15) == 0 && (dbias_dtype == MOBGT_F32 || layer_stride % 8 == 0), MOBGT_ERR_BAD_SHAPE,
                  "mobgt_bias_direct_bwd: dBias planes must be 16-byte aligned");
    const K2Common c{n, sq_off, rel_pos, poi_pos, nullptr, B, T, Tp, 0, rel_pos_max, 0};
    auto f = H == 8 ? bias_direct_bwd<8> : bias_direct_bwd<12>;
    return f(c, feat, num_bins, dBias, dbias_dtype, n_layers, layer_stride, workspace, workspace_bytes, dR, dPpos, dE, dtvd,
             static_cast<cudaStream_t>(stream));
}
