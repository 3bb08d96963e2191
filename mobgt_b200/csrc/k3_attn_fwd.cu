// K3 (forward) — biased multi-head attention on tcgen05 / TMEM, fed by TMA (sm_100a).
//
// Replaces MultiHeadAttention.forward's core, model_fqandtoyo.py:1693-1706:
//     q = q * scale ; x = q @ k^T + attn_bias ; x = softmax(x, dim=3) ; x = x @ v
// for PACKED (var-len) graphs: graph g owns token rows tok_off[g] .. tok_off[g+1].  The padding-column
// mask (the -inf columns of collator.py:57-64) is applied in-tile from the sequence lengths, the bias tile is
// streamed by TMA, and the scores never touch HBM.
//
// One CTA per (graph, head); K and V of the graph stay resident in shared memory.
//   S  = Q_i K_j^T      tcgen05.mma  M=128, N<=128, K=dp                          -> TMEM cols [0,128)
//   P  = softmax tile   tcgen05.ld -> registers (+ bias tile from smem, online max/sum) -> bf16 -> smem
//   O += P V_j          tcgen05.mma  M=128, N=dp, K=kv                             -> TMEM cols [128,128+dp)
// The head dim d is a template parameter, built for 24 (dp = 32: one zero K-padding chunk, two K=16 MMAs for S) and
// 16 (dp = 16: no padding, one MMA for S); k3_small.cuh AttnShape.
// Operands use the no-swizzle [chunk][row][8] layout of umma.cuh (3-D TMA boxes {8, 128 rows, d/8 chunks});
// the bias tile is two {64 x 128} boxes with the 128-byte TMA swizzle.
#include <cuda_bf16.h>

#include "common.cuh"
#include "k3_small.cuh"
#include "umma.cuh"

namespace mobgt {
using namespace sm100;

constexpr int kTile = 128;       // query rows per tile == KV rows per box
constexpr int kBiasTileBytes = 2 * kTile * 128;  // two 64-column halves, 128 B per row
constexpr int kPBytes = 16 * kTile * 16;         // [16 chunks][128 rows][16 B]

struct AttnFwdParams {
    const int32_t *tok_off;  // [B+1]
    __nv_bfloat16 *out;      // [Ntok, H*d]
    float *lse;              // [Ntok, H]
    int H;
    float scale;
    int max_boxes;           // ceil(Tmax / 128): K/V boxes provisioned in shared memory
    long long *timeline;     // debug (mobgt_debug_set_timeline) or NULL
    AttnDrop drop;           // attention dropout on P (model_fqandtoyo.py:1704); th16 == 0 in eval
    const __nv_bfloat16 *q, *k, *v;   // raw views of the operands (row stride qkv_stride) for the single-token tail
    int64_t qkv_stride;
    const __nv_bfloat16 *bias;        // [B,H,T,Tp]
    int T, Tp;
    int small_t;                      // graphs of at most this many tokens belong to the SIMT kernel (k3_attn_small.cu); 0: none
    const int32_t *order;             // [B] graph ids in launch order (descending size) or NULL
    int n_items;                      // B * H work items; CTA b works on items b, b + gridDim.x, ... (persistent CTAs)
    int large_t;                      // graphs of more tokens belong to the SIMT kernel of k3_attn_large.cu
};

// the d bf16 of row `row` of a [chunk][row][8] operand box -> fp32
template <int kD>
__device__ __forceinline__ void fwd_box_row(const uint8_t *box, int row, float (&f)[kD]) {
    uint4 w[kD / 8];
#pragma unroll
    for (int c = 0; c < kD / 8; ++c) w[c] = *reinterpret_cast<const uint4 *>(box + c * (kTile * 16) + row * 16);
    unpack_words<kD / 8>(w, f);
}

__device__ __forceinline__ float fast_exp2(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

// 256 threads = two warpgroups.  Thread (wg, t128) owns query row t128 of the current tile (TMEM lane t128; warps w and
// w+4 may both access lanes 32*(w%4)..+31) and the 16-column chunks c0 = 16*wg, 16*wg + 32, ... of the score tile, i.e. at
// most 64 scores, which stay in registers between the max pass and the exp pass (one TMEM read, one bias decode).
// The row max is exchanged between the warpgroups through shared memory; the row sums are combined once per query tile.
// After the max pass nobody needs the bias tile any more, so the next tile's TMA load is issued there and overlaps the
// exp pass and the P.V MMA.
// kDrop: training-mode attention dropout — the row sum (softmax denominator) is taken BEFORE the mask, the bf16 P tile that
// feeds the P.V MMA holds only the kept probabilities, and 1 / (1 - p) is folded into the final 1 / l normalisation.
//
// Single-token tail ("fold"): a graph of 128 m + 1 tokens (n = 128 m nodes + the graph token) runs the MMA loop over its
// m x m full tiles only; the last token sp = 128 m is handled by SIMT: its key column enters every row's online softmax as
// one more (register) block in the tile epilogue, and its own query row is one block-wide softmax + a small mat-vec.
template <int kAttD, bool kDrop>
__global__ void __launch_bounds__(256, 2)
k3_attn_fwd_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmK,
                   const __grid_constant__ CUtensorMap tmV, const __grid_constant__ CUtensorMap tmBias,
                   const AttnFwdParams p) {
    extern __shared__ __align__(1024) uint8_t smem[];
    __shared__ __align__(8) uint64_t bar_q, bar_kv, bar_bias, bar_s, bar_o;
    __shared__ uint32_t tmem_slot;
    __shared__ float sMax[2][kTile];
    __shared__ float sTail[4 * kTile];          // fold: score (log2 units) of (row r, key sp)
    __shared__ float sTp[4 * kTile + 4];        // fold: kept probabilities of (row sp, key c)
    __shared__ float sSp[3][kAttD];             // fold: q, k, v of token sp
    __shared__ float sRed[AttnShape<kAttD>::kSegs][kAttD];
    __shared__ float sScal[16];
    using Sh = AttnShape<kAttD>;
    constexpr int kAttChunks = Sh::kChunks, kDPad = Sh::kDPad, kBoxBytes = Sh::kBoxBytes, kBoxTxBytes = Sh::kBoxTxBytes;
    constexpr int kSegs = Sh::kSegs;

    MOBGT_STAMP(p.timeline, 0);
    const int tid = threadIdx.x, warp = tid >> 5, wg = tid >> 7, t128 = tid & 127;
    const bool warp0 = warp_index_uniform() == 0;   // the issuing warp (one elected lane issues TMA / MMA)
    // ---- persistent CTA: work item = (graph, head) in launch order; items of small graphs (SIMT kernel) are skipped.
    // next_item: the first item >= `from` (stepping by the grid) that this kernel owns, with its header.
    struct Item { int idx, g, h, t0, Tg; };
    auto next_item = [&](int from) -> Item {
        Item it{from, 0, 0, 0, 0};
        for (; it.idx < p.n_items; it.idx += (int)gridDim.x) {
            const int gi = it.idx / p.H;
            it.h = it.idx - gi * p.H;
            it.g = p.order ? p.order[gi] : gi;      // largest graphs first
            it.t0 = p.tok_off[it.g];
            it.Tg = p.tok_off[it.g + 1] - it.t0;
            if (it.Tg > p.small_t && it.Tg <= p.large_t) break;
        }
        return it;
    };
    Item cur = next_item((int)blockIdx.x);
    if (cur.idx >= p.n_items) return;                      // the whole CTA: nothing has been set up yet
    uint8_t *sBias = smem + ((1024u - (smem_u32(smem) & 1023u)) & 1023u);   // 32 KB, 1024-aligned (swizzle atom)
    uint8_t *sP = sBias + kBiasTileBytes;                    // 32 KB
    uint8_t *sQ = sP + kPBytes;                              // 8 KB
    uint8_t *sK = sQ + kBoxBytes;                            // max_boxes * 8 KB
    uint8_t *sV = sK + (size_t)p.max_boxes * kBoxBytes;      // max_boxes * 8 KB

    if (tid == 0) {
        mbar_init(&bar_q, 1);
        mbar_init(&bar_kv, 1);
        mbar_init(&bar_bias, 1);
        mbar_init(&bar_s, 1);
        mbar_init(&bar_o, 1);
        fence_barrier_init();
        tma_prefetch_desc(&tmQ);
        tma_prefetch_desc(&tmK);
        tma_prefetch_desc(&tmV);
        tma_prefetch_desc(&tmBias);
    }
    // zero the K-padding chunk (d = 24..31) of Q and of every K / V box: 128 rows x 16 B each (d = 16: no padding)
    if (kDPad != kAttD) {
        const uint4 z = make_uint4(0, 0, 0, 0);
        if (wg == 0) *reinterpret_cast<uint4 *>(sQ + 3 * kTile * 16 + t128 * 16) = z;
        uint8_t *kv = wg == 0 ? sK : sV;
        for (int b = 0; b < p.max_boxes; ++b) *reinterpret_cast<uint4 *>(kv + (size_t)b * kBoxBytes + 3 * kTile * 16 + t128 * 16) = z;
    }
    if (warp == 0) tmem_alloc<256>(&tmem_slot);
    fence_proxy_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    MOBGT_STAMP(p.timeline, 1);
    const uint32_t tmem = tmem_slot;
    const uint32_t tS = tmem, tO = tmem + 128;
    const uint32_t lane_off = (uint32_t)((warp & 3) * 32) << 16;
    const float sl2 = p.scale * 1.4426950408889634f;  // scale * log2(e)
    constexpr float kL2e = 1.4426950408889634f;
    uint32_t seed_lo = 0, seed_hi = 0;
    if (kDrop) attn_drop_fold_seed(p.drop, seed_lo, seed_hi);
    const uint32_t th_hi = p.drop.th16 << 16;

    // the first loads of an item (thread 0 only): all K / V boxes, query tile 0, bias tile (0, 0).  For the CTA's first item
    // they are issued here; for every later item at the end of its predecessor (the operands' shared memory is free once the
    // last P.V MMA has completed), so they fly under the predecessor's epilogue and the barrier / TMEM set-up is paid once.
    auto load_item = [&](const Item &it) {
        const bool ifold = it.Tg > kTile && (it.Tg % kTile) == 1;
        const int inb = ifold ? it.Tg / kTile : ceil_div(it.Tg, kTile);
        mbar_expect_tx(&bar_kv, (uint32_t)(2 * inb * kBoxTxBytes));
        for (int b = 0; b < inb; ++b) {
            tma_load_3d(sK + (size_t)b * kBoxBytes, &tmK, &bar_kv, 0, it.t0 + b * kTile, it.h * kAttChunks);
            tma_load_3d(sV + (size_t)b * kBoxBytes, &tmV, &bar_kv, 0, it.t0 + b * kTile, it.h * kAttChunks);
        }
        mbar_expect_tx(&bar_q, kBoxTxBytes);
        tma_load_3d(sQ, &tmQ, &bar_q, 0, it.t0, it.h * kAttChunks);
        mbar_expect_tx(&bar_bias, kBiasTileBytes);
        tma_load_3d(sBias, &tmBias, &bar_bias, 0, 0, it.g * p.H + it.h);
        tma_load_3d(sBias + kTile * 128, &tmBias, &bar_bias, 64, 0, it.g * p.H + it.h);
    };
    if (tid == 0) load_item(cur);
    uint32_t ph_bias = 0, ph_s = 0, ph_o = 0, ph_kv = 0, nq = 0;   // barrier phases run on across the items (nq: Q tiles loaded so far)

  while (cur.idx < p.n_items) {
    const int g = cur.g, h = cur.h, t0 = cur.t0, Tg = cur.Tg;
    const bool fold = Tg > kTile && (Tg % kTile) == 1;     // single-token tail handled by SIMT (see above)
    const int NB = fold ? Tg / kTile : ceil_div(Tg, kTile);
    const int sp = Tg - 1;                                 // the tail token (fold only)
    const int plane = g * p.H + h;

    // fold: the bias row / column of the tail token and its q, k, v — global loads issued at the very top of the item
    float b_row[3] = {0.f, 0.f, 0.f}, b_col[2] = {0.f, 0.f};
    if (fold) {
        const __nv_bfloat16 *bias_pl0 = p.bias + (size_t)plane * p.T * p.Tp;
#pragma unroll
        for (int u = 0; u < 3; ++u)
            if (tid + u * 256 < Tg) b_row[u] = __bfloat162float(bias_pl0[(size_t)sp * p.Tp + tid + u * 256]);
#pragma unroll
        for (int u = 0; u < 2; ++u)
            if (tid + u * 256 < sp) b_col[u] = __bfloat162float(bias_pl0[(size_t)(tid + u * 256) * p.Tp + sp]);
    }
    if (fold && tid < 3 * kAttD) {   // q, k, v of the tail token as fp32
        const int which = tid / kAttD, e = tid - which * kAttD;
        const __nv_bfloat16 *src = which == 0 ? p.q : which == 1 ? p.k : p.v;
        sSp[which][e] = __bfloat162float(src[(size_t)(t0 + sp) * p.qkv_stride + h * kAttD + e]);
    }
    const Item nxt = next_item(cur.idx + (int)gridDim.x);   // its header is needed by thread 0 at the end of this item
    __syncthreads();                                        // sSp of this item is visible

    auto load_bias = [&](int i, int j) {   // thread 0 only
        mbar_expect_tx(&bar_bias, kBiasTileBytes);
        tma_load_3d(sBias, &tmBias, &bar_bias, j * kTile, i * kTile, plane);
        tma_load_3d(sBias + kTile * 128, &tmBias, &bar_bias, j * kTile + 64, i * kTile, plane);
    };
    auto load_q = [&](int i) {             // thread 0 only
        mbar_expect_tx(&bar_q, kBoxTxBytes);
        tma_load_3d(sQ, &tmQ, &bar_q, 0, t0 + i * kTile, h * kAttChunks);
    };
    // S = Q_i K_j^T into TMEM (thread 0 only); new_q: first block of a query tile -> wait for its Q box
    auto issue_s = [&](int j, int new_q_tile) {   // new_q_tile >= 0: first block of that query tile -> wait for its Q box
        if (new_q_tile >= 0) mbar_wait(&bar_q, (nq + (uint32_t)new_q_tile) & 1u);
        const int nbj = round_up(min(kTile, Tg - j * kTile), 16);
        const uint32_t idesc = make_idesc_bf16(kTile, nbj, 0, 0);
        const uint32_t aq = smem_u32(sQ), bk = smem_u32(sK + (size_t)j * kBoxBytes);
#pragma unroll
        for (int ks = 0; ks < kDPad / 16; ++ks)
            umma_bf16(tS, make_smem_desc(aq + ks * 2 * kTile * 16, kTile * 16, 128),
                      make_smem_desc(bk + ks * 2 * kTile * 16, kTile * 16, 128), idesc, ks > 0);
        umma_commit(&bar_s);
    };
    if (warp0 && elect_one()) {
        mbar_wait(&bar_kv, ph_kv);
        tc_fence_after();
        MOBGT_STAMP(p.timeline, 2);
        issue_s(0, 0);
        MOBGT_STAMP(p.timeline, 3);
    }
    __syncwarp();

    if (fold) {   // ---- the single-token tail, SIMT (overlaps the first S MMA)
        const __nv_bfloat16 *bias_pl = p.bias + (size_t)plane * p.T * p.Tp;
        mbar_wait(&bar_kv, ph_kv);                  // K / V boxes and the first Q tile have landed
        mbar_wait(&bar_q, nq & 1u);                 // (tile 0 stays put until the loop)
        // (1) every full-tile row r against key sp: the score joins the row's online softmax in the tile epilogue
#pragma unroll
        for (int u = 0; u < 2; ++u) {
            const int r = tid + u * 256;
            if (r >= sp) break;
            float qf[kAttD];
            if (r < kTile) {      // tile 0: from shared memory
                fwd_box_row<kAttD>(sQ, r, qf);
            } else {
                const uint4 *qg = reinterpret_cast<const uint4 *>(p.q + (size_t)(t0 + r) * p.qkv_stride + h * kAttD);
                uint4 w[kAttChunks];
#pragma unroll
                for (int c = 0; c < kAttChunks; ++c) w[c] = qg[c];
                unpack_words<kAttChunks>(w, qf);
            }
            float dot = 0.f;
#pragma unroll
            for (int e = 0; e < kAttD; ++e) dot = fmaf(qf[e], sSp[1][e], dot);
            sTail[r] = fmaf(dot, sl2, b_col[u] * kL2e);
        }
        // (2) query row sp against every key: block-wide softmax
        float sc[3], mx = -INFINITY;
#pragma unroll
        for (int u = 0; u < 3; ++u) {
            const int c = tid + u * 256;
            sc[u] = -INFINITY;
            if (c < Tg) {
                float dot = 0.f;
                if (c < sp) {
                    float kf[kAttD];
                    fwd_box_row<kAttD>(sK + (size_t)(c >> 7) * kBoxBytes, c & 127, kf);
#pragma unroll
                    for (int e = 0; e < kAttD; ++e) dot = fmaf(sSp[0][e], kf[e], dot);
                } else {
#pragma unroll
                    for (int e = 0; e < kAttD; ++e) dot = fmaf(sSp[0][e], sSp[1][e], dot);
                }
                sc[u] = fmaf(dot, sl2, b_row[u] * kL2e);
                mx = fmaxf(mx, sc[u]);
            }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
        if ((tid & 31) == 0) sScal[warp] = mx;
        __syncthreads();
        mx = sScal[0];
#pragma unroll
        for (int w8 = 1; w8 < 8; ++w8) mx = fmaxf(mx, sScal[w8]);
        const uint32_t rk = kDrop ? attn_drop_rowkey((uint32_t)plane, (uint32_t)sp, seed_lo, seed_hi) : 0u;
        float ls = 0.f;
#pragma unroll
        for (int u = 0; u < 3; ++u) {
            const int c = tid + u * 256;
            if (c < Tg) {
                const float pe = fast_exp2(sc[u] - mx);
                ls += pe;                                   // the denominator is taken before the dropout mask
                bool kp = true;
                if (kDrop) kp = (attn_drop_keep8(rk, (uint32_t)(c >> 3), p.drop.th16) >> (c & 7)) & 1u;
                sTp[c] = kp ? pe : 0.f;
            }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) ls += __shfl_xor_sync(0xffffffffu, ls, o);
        if ((tid & 31) == 0) sScal[8 + warp] = ls;
        __syncthreads();
        ls = 0.f;
#pragma unroll
        for (int w8 = 0; w8 < 8; ++w8) ls += sScal[8 + w8];
        if (tid < 240) {   // O[sp] = sum_c P[c] v_c : thread = (e, seg)
            const int seg = tid / kAttD, e = tid - seg * kAttD;
            float a = 0.f;
            for (int c = seg; c < sp; c += kSegs) {
                const __nv_bfloat16 *vb = reinterpret_cast<const __nv_bfloat16 *>(
                    sV + (size_t)(c >> 7) * kBoxBytes + (e >> 3) * (kTile * 16) + (c & 127) * 16) + (e & 7);
                a = fmaf(sTp[c], __bfloat162float(*vb), a);
            }
            sRed[seg][e] = a;
        }
        __syncthreads();
        if (tid < kAttD) {
            float a = sTp[sp] * sSp[2][tid];
#pragma unroll
            for (int sg = 0; sg < kSegs; ++sg) a += sRed[sg][tid];
            p.out[(size_t)(t0 + sp) * (p.H * kAttD) + h * kAttD + tid] = __float2bfloat16_rn(a * (kDrop ? p.drop.inv_keep : 1.0f) / ls);
            if (tid == 0) p.lse[(size_t)(t0 + sp) * p.H + h] = (mx + log2f(ls)) * 0.6931471805599453f;
        }
    }

    for (int i = 0; i < NB; ++i) {
        const int row = i * kTile + t128;      // query row inside the graph
        const uint32_t rowkey = kDrop ? attn_drop_rowkey((uint32_t)plane, (uint32_t)row, seed_lo, seed_hi) : 0u;
        const bool row_ok = row < Tg;
        const bool warp_live = i * kTile + (warp & 3) * 32 < Tg;   // any valid query row in this warp's 32 lanes?
        float m_run = -INFINITY, l_run = 0.f;  // running max (log2 units of the scaled score); this warpgroup's share of the sum
        for (int j = 0; j < NB; ++j) {
            const int kv_valid = min(kTile, Tg - j * kTile);    // valid key columns in this block
            const int nb = round_up(kv_valid, 16);              // MMA N / K extent
            __syncwarp();
            mbar_wait(&bar_s, ph_s);
            ph_s ^= 1;
            MOBGT_STAMP(p.timeline, 8 + 8 * (i * NB + j) + 0);   // S ready
            if (j + 1 == NB && i + 1 < NB && warp0 && elect_one()) load_q(i + 1);   // the last S MMA of this tile has consumed Q
            mbar_wait(&bar_bias, ph_bias);
            ph_bias ^= 1;
            tc_fence_after();
            MOBGT_STAMP(p.timeline, 8 + 8 * (i * NB + j) + 1);   // bias tile ready

            // ---- pass 1: s = scale * S + bias (log2 units) for this thread's columns -> registers; row max
            uint32_t sv[4][16];           // raw S, then (in place) the biased scores: the only per-tile register array
            float m_blk = -INFINITY;
            if (warp_live) {
#pragma unroll
                for (int cc = 0; cc < 4; ++cc)
                    if (wg * 16 + cc * 32 < nb) tmem_ld16(tS + lane_off + wg * 16 + cc * 32, sv[cc]);   // all loads in flight
                tmem_ld_wait();
#pragma unroll
                for (int cc = 0; cc < 4; ++cc) {
                    const int c0 = wg * 16 + cc * 32;
                    if (c0 < nb) {
#pragma unroll
                        for (int q8 = 0; q8 < 2; ++q8) {
                            const int c8 = (c0 >> 3) + q8;             // 8-column chunk index inside the 128-wide tile
                            const uint8_t *bp = sBias + (c8 >> 3) * (kTile * 128) + t128 * 128 + (((c8 & 7) ^ (t128 & 7)) << 4);
                            uint4 bv = *reinterpret_cast<const uint4 *>(bp);
                            if (!row_ok) bv = make_uint4(0, 0, 0, 0);   // bias rows past the graph are never written
                            const uint32_t bw[4] = {bv.x, bv.y, bv.z, bv.w};
                            const bool full = c8 * 8 + 8 <= kv_valid;
#pragma unroll
                            for (int e = 0; e < 8; ++e) {
                                const float bias = __uint_as_float((e & 1) ? (bw[e >> 1] & 0xFFFF0000u) : (bw[e >> 1] << 16));
                                float s = fmaf(__uint_as_float(sv[cc][q8 * 8 + e]), sl2, bias * kL2e);
                                if (!full && c8 * 8 + e >= kv_valid) s = -INFINITY;   // padding key columns (collator.py:57-64)
                                sv[cc][q8 * 8 + e] = __float_as_uint(s);
                                m_blk = fmaxf(m_blk, s);
                            }
                        }
                    }
                }
            }
            MOBGT_STAMP(p.timeline, 8 + 8 * (i * NB + j) + 2);   // pass 1 done (thread 0)
            sMax[wg][t128] = m_blk;
            tc_fence_before();            // this thread's tcgen05.ld of S precede the next S MMA issued after the barrier
            __syncthreads();              // both halves of every row max are visible; nobody reads the bias tile any more
            if (warp0 && elect_one()) {   // every thread holds its scores in registers: TMEM S and the bias tile are free again
                tc_fence_after();
                if (j + 1 < NB) {
                    load_bias(i, j + 1);
                    issue_s(j + 1, -1);
                } else if (i + 1 < NB) {
                    load_bias(i + 1, 0);
                    issue_s(0, i + 1);
                }
            }
            MOBGT_STAMP(p.timeline, 8 + 8 * (i * NB + j) + 3);   // barrier A passed, next loads / S MMA issued
            m_blk = fmaxf(m_blk, sMax[wg ^ 1][t128]);
            const float m_new = fmaxf(m_run, m_blk);
            const float m_use = (m_new == -INFINITY) ? 0.f : m_new;   // rows past the graph: keep the arithmetic finite
            const float alpha = (j == 0) ? 0.f : fast_exp2(m_run - m_use);
            // ---- pass 2: p = 2^(s - m), row sum, bf16 P tile to shared memory ([chunk][row][8])
            if (j > 0) {   // the previous P.V must be complete before P / O are touched again
                mbar_wait(&bar_o, ph_o);
                ph_o ^= 1;
                tc_fence_after();
            }
            float l_blk = 0.f;
            if (warp_live) {
#pragma unroll
                for (int cc = 0; cc < 4; ++cc) {
                    const int c0 = wg * 16 + cc * 32;
                    if (c0 < nb) {
#pragma unroll
                        for (int q8 = 0; q8 < 2; ++q8) {
                            const int c8 = (c0 >> 3) + q8;
                            float pv[8];
#pragma unroll
                            for (int e = 0; e < 8; ++e) {
                                pv[e] = fast_exp2(__uint_as_float(sv[cc][q8 * 8 + e]) - m_use);
                                l_blk += pv[e];     // row sum in fp32 (P is rounded to bf16 only for the tensor-core operand)
                            }
                            if (kDrop) {
                                const AttnDropWords dw = attn_drop_words(rowkey, (uint32_t)(j * (kTile / 8) + c8));
#pragma unroll
                                for (int e = 0; e < 8; ++e) pv[e] = attn_drop_keep(dw, e, th_hi) ? pv[e] : 0.f;
                            }
                            uint4 pk;
                            pk.x = pack_bf16(pv[0], pv[1]);
                            pk.y = pack_bf16(pv[2], pv[3]);
                            pk.z = pack_bf16(pv[4], pv[5]);
                            pk.w = pack_bf16(pv[6], pv[7]);
                            *reinterpret_cast<uint4 *>(sP + c8 * (kTile * 16) + t128 * 16) = pk;
                        }
                    }
                }
            }
            l_run = l_run * alpha + l_blk;
            m_run = m_new;
            if (j > 0 && warp_live && (kDPad == 32 || wg == 0)) {   // rescale the running O accumulator (columns [16 wg, 16 wg + 16))
                uint32_t ov[16];
                tmem_ld16(tO + lane_off + wg * 16, ov);
                tmem_ld_wait();
#pragma unroll
                for (int e = 0; e < 16; ++e) ov[e] = __float_as_uint(__uint_as_float(ov[e]) * alpha);
                tmem_st16(tO + lane_off + wg * 16, ov);
                tmem_st_wait();
            }
            MOBGT_STAMP(p.timeline, 8 + 8 * (i * NB + j) + 4);   // pass 2 done (thread 0)
            fence_proxy_async_smem();
            tc_fence_before();
            __syncthreads();
            MOBGT_STAMP(p.timeline, 8 + 8 * (i * NB + j) + 5);   // barrier B passed
            if (warp0 && elect_one()) {
                tc_fence_after();
                const uint32_t idesc = make_idesc_bf16(kTile, kDPad, 0, 1);
                const uint32_t ap = smem_u32(sP), bv = smem_u32(sV + (size_t)j * kBoxBytes);
                for (int ks = 0; ks < nb / 16; ++ks)
                    umma_bf16(tO, make_smem_desc(ap + ks * 2 * kTile * 16, kTile * 16, 128),
                              make_smem_desc(bv + ks * 256, 128, kTile * 16), idesc, (j > 0 || ks > 0));
                umma_commit(&bar_o);
            }
            __syncwarp();
        }
        // ---- epilogue of the query tile: O / l -> bf16, lse.  The two warpgroups' shares of the row sum are exchanged
        //      through sMax (free since the last barrier of the j loop); warpgroup wg stores O columns [16 wg, 16 wg + 16) < d.
        sMax[wg][t128] = l_run;
        mbar_wait(&bar_o, ph_o);
        ph_o ^= 1;
        tc_fence_after();
        // last query tile: every MMA of this item has completed and the bias tile was consumed in pass 1, so K / V / Q / bias
        // shared memory is free: the next item's first loads start now and fly under this epilogue
        if (i + 1 == NB && tid == 0 && nxt.idx < p.n_items) load_item(nxt);
        __syncthreads();
        if (warp_live && (kAttD > 16 || wg == 0)) {
            uint32_t ov[16];
            tmem_ld16(tO + lane_off + wg * 16, ov);
            tmem_ld_wait();
            if (row_ok) {
                float l_tot = sMax[0][t128] + sMax[1][t128];
                if (fold) {   // one more online-softmax block: the tail key's column
                    const float st = sTail[row];
                    const float m_new = fmaxf(m_run, st);
                    const float al = fast_exp2(m_run - m_new), pe = fast_exp2(st - m_new);
                    l_tot = fmaf(l_tot, al, pe);
                    bool kp = true;
                    if (kDrop) kp = (attn_drop_keep8(rowkey, (uint32_t)(sp >> 3), p.drop.th16) >> (sp & 7)) & 1u;
                    const float pd = kp ? pe : 0.f;
#pragma unroll
                    for (int e = 0; e < 16; ++e)
                        if (wg == 0 || e < kAttD - 16)
                            ov[e] = __float_as_uint(fmaf(__uint_as_float(ov[e]), al, pd * sSp[2][wg * 16 + e]));
                    m_run = m_new;
                }
                const float inv = (kDrop ? p.drop.inv_keep : 1.0f) / l_tot;
                uint32_t w[8];
#pragma unroll
                for (int e = 0; e < 8; ++e)
                    w[e] = pack_bf16(__uint_as_float(ov[2 * e]) * inv, __uint_as_float(ov[2 * e + 1]) * inv);
                uint4 *dst = reinterpret_cast<uint4 *>(p.out + (size_t)(t0 + row) * (p.H * kAttD) + h * kAttD);
                if (wg == 0) {
                    dst[0] = make_uint4(w[0], w[1], w[2], w[3]);
                    dst[1] = make_uint4(w[4], w[5], w[6], w[7]);
                    p.lse[(size_t)(t0 + row) * p.H + h] = (m_run + log2f(l_tot)) * 0.6931471805599453f;
                } else {
                    dst[2] = make_uint4(w[0], w[1], w[2], w[3]);   // d = 24: columns 16..23 (24..31 are the MMA padding)
                }
            }
        }
        MOBGT_STAMP(p.timeline, 8 + 8 * (i * NB + NB - 1) + 7);   // tile epilogue done
        tc_fence_before();
        __syncthreads();   // every thread is done with TMEM S/O before the next tile's MMAs
    }
    ph_kv ^= 1u;
    nq += (uint32_t)NB;
    cur = nxt;
  }   // items
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc<256>(tmem);
    MOBGT_STAMP(p.timeline, 4);
}

}  // namespace mobgt

using namespace mobgt;

namespace {
// qkv: three bf16 matrices of [ntok, H*d] with a common row stride (elements); typically slices of one fused
// [ntok, 3*H*d] projection.  bias: bf16 [B, H, T, Tp].  out: bf16 [ntok, H*d] (contiguous).  lse: f32 [ntok, H].
template <int kAttD>
int32_t attn_fwd(const void *q, const void *k, const void *v, int64_t qkv_row_stride, const void *bias,
                 const int32_t *tok_off, const int32_t *graph_order, int32_t B, int32_t H, int32_t ntok,
                 int32_t T, int32_t Tp, int32_t t_max_host, int32_t t_min_host, float scale, float drop_p, uint64_t seed,
                 const void *seed_dev, void *out, float *lse, void *stream) {
    using Sh = AttnShape<kAttD>;
    constexpr int kAttChunks = Sh::kChunks, kBoxBytes = Sh::kBoxBytes;
    MOBGT_REQUIRE(q && k && v && bias && tok_off && out && lse, MOBGT_ERR_NULL, "mobgt_attn_fwd: null pointer");
    MOBGT_REQUIRE(H >= 1 && B >= 0 && ntok >= 0, MOBGT_ERR_BAD_SHAPE, "mobgt_attn_fwd: B=%d H=%d ntok=%d", B, H, ntok);
    MOBGT_REQUIRE(qkv_row_stride % 8 == 0 && Tp % 8 == 0 && Tp >= T, MOBGT_ERR_BAD_SHAPE,
                  "mobgt_attn_fwd: row stride %lld and Tp=%d must be multiples of 8", (long long)qkv_row_stride, Tp);
    MOBGT_REQUIRE(t_max_host >= 1 && t_max_host <= T && T <= MOBGT_MAX_MODEL_NODES + 1, MOBGT_ERR_BAD_SHAPE,
                  "mobgt_attn_fwd: t_max=%d T=%d (T <= 1025: graphs of at most 1024 nodes)", t_max_host, T);
    MOBGT_REQUIRE(drop_p >= 0.f && drop_p < 1.f, MOBGT_ERR_BAD_SHAPE, "mobgt_attn_fwd: drop_p=%f must be in [0, 1)", drop_p);
    if (B == 0 || ntok == 0) return MOBGT_OK;
    // graphs of <= kSmallT tokens: SIMT kernel; the others: tensor cores.  Both kernels select their graphs on the device, so
    // the host only decides which launches can be skipped (t_min_host = 0: unknown, e.g. a CUDA graph shared by many batches).
    const bool any_small = (t_min_host <= 0 || t_min_host <= kSmallT) && H % 4 == 0;
    const bool any_large = t_max_host > kSmallT;
    ForkJoin fj{};
    bool forked = false;
    if (any_small) {
        SmallAttnParams sp{};
        sp.tok_off = tok_off;
        sp.order = graph_order;
        sp.q = static_cast<const __nv_bfloat16 *>(q); sp.k = static_cast<const __nv_bfloat16 *>(k); sp.v = static_cast<const __nv_bfloat16 *>(v);
        sp.qkv_stride = qkv_row_stride;
        sp.bias = static_cast<const __nv_bfloat16 *>(bias);
        sp.H = H; sp.T = T; sp.Tp = Tp; sp.scale = scale; sp.small_t = kSmallT;
        sp.drop = make_attn_drop(drop_p, seed, seed_dev);
        sp.out = static_cast<__nv_bfloat16 *>(out); sp.lse = lse;
        if (!any_large) return launch_small_attn_fwd<kAttD>(sp, B, static_cast<cudaStream_t>(stream));
        // both kernels: they work on disjoint graphs, so the SIMT one runs on a side stream next to the tensor-core one
        int32_t rc = get_fork_join(0, &fj);
        if (rc) return rc;
        MOBGT_CUDA_OK(cudaEventRecord(fj.fork, static_cast<cudaStream_t>(stream)));
        MOBGT_CUDA_OK(cudaStreamWaitEvent(fj.side, fj.fork, 0));
        rc = launch_small_attn_fwd<kAttD>(sp, B, fj.side);
        MOBGT_CUDA_OK(cudaEventRecord(fj.join, fj.side));
        forked = true;
        if (rc) {
            cudaStreamWaitEvent(static_cast<cudaStream_t>(stream), fj.join, 0);
            return rc;
        }
    }
    auto run_tensor_core = [&]() -> int32_t {
    if (t_min_host > kLargeT) return MOBGT_OK;    // every graph is a large one
    CUtensorMap tmQ, tmK, tmV, tmB;
    const void *ptrs[3] = {q, k, v};
    CUtensorMap *maps[3] = {&tmQ, &tmK, &tmV};
    for (int i = 0; i < 3; ++i) {
        uint64_t dims[3] = {8, (uint64_t)ntok, (uint64_t)H * kAttChunks};
        uint64_t str[2] = {(uint64_t)qkv_row_stride * 2, 16};
        uint32_t box[3] = {8, kTile, kAttChunks};
        int32_t rc = encode_tmap_bf16(maps[i], ptrs[i], 3, dims, str, box, 0);
        if (rc) return rc;
    }
    {
        uint64_t dims[3] = {(uint64_t)Tp, (uint64_t)T, (uint64_t)B * H};
        uint64_t str[2] = {(uint64_t)Tp * 2, (uint64_t)T * Tp * 2};
        uint32_t box[3] = {64, kTile, 1};
        int32_t rc = encode_tmap_bf16(&tmB, bias, 3, dims, str, box, 1);
        if (rc) return rc;
    }
    // a graph of 128 m + 1 tokens keeps only its m full boxes in shared memory (single-token tail); this kernel's graphs have
    // at most kLargeT = 513 tokens
    const int t_tc = min(t_max_host, kLargeT);
    const int max_boxes = t_tc > kTile && t_tc % kTile == 1 ? t_tc / kTile : ceil_div(t_tc, kTile);
    const size_t smem = (size_t)kBiasTileBytes + kPBytes + kBoxBytes + (size_t)2 * max_boxes * kBoxBytes + 1024;
    AttnFwdParams p{tok_off, static_cast<__nv_bfloat16 *>(out), lse, H, scale, max_boxes, g_timeline_dev,
                    make_attn_drop(drop_p, seed, seed_dev),
                    static_cast<const __nv_bfloat16 *>(q), static_cast<const __nv_bfloat16 *>(k),
                    static_cast<const __nv_bfloat16 *>(v), qkv_row_stride, static_cast<const __nv_bfloat16 *>(bias), T, Tp,
                    any_small ? kSmallT : 0, graph_order, B * H, kLargeT};
    auto kern = p.drop.th16 ? k3_attn_fwd_kernel<kAttD, true> : k3_attn_fwd_kernel<kAttD, false>;
    MOBGT_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int grid = B * H < 2 * kNumSMs ? B * H : 2 * kNumSMs;     // persistent: two CTAs per SM, each loops over its items
    kern<<<grid, 256, smem, static_cast<cudaStream_t>(stream)>>>(tmQ, tmK, tmV, tmB, p);
    MOBGT_LAUNCH_OK("k3_attn_fwd_kernel");
    return MOBGT_OK;
    };
    int32_t rc = run_tensor_core();
    if (rc == MOBGT_OK && t_max_host > kLargeT) {   // graphs of 514 .. 1025 tokens
        LargeAttnParams lp{};
        lp.tok_off = tok_off; lp.order = graph_order; lp.q = q; lp.k = k; lp.v = v; lp.qkv_stride = qkv_row_stride; lp.bias = bias;
        lp.H = H; lp.T = T; lp.Tp = Tp; lp.scale = scale; lp.t_lo = kLargeT; lp.drop = make_attn_drop(drop_p, seed, seed_dev);
        lp.out = out; lp.lse = lse;
        rc = launch_large_attn_fwd<__nv_bfloat16, kAttD>(lp, B, t_max_host, static_cast<cudaStream_t>(stream));
    }
    if (forked) cudaStreamWaitEvent(static_cast<cudaStream_t>(stream), fj.join, 0);   // join on every path
    return rc;
}
}  // namespace

extern "C" int32_t mobgt_attn_fwd_hd(const void *q, const void *k, const void *v, int64_t qkv_row_stride, const void *bias,
                                     const int32_t *tok_off, const int32_t *graph_order, int32_t B, int32_t H, int32_t ntok,
                                     int32_t T, int32_t Tp, int32_t t_max_host, int32_t t_min_host, float scale, float drop_p,
                                     uint64_t seed, const void *seed_dev, void *out, float *lse, int32_t head_dim, void *stream) {
    MOBGT_REQUIRE(head_dim == 16 || head_dim == 24, MOBGT_ERR_UNSUPPORTED,
                  "mobgt_attn_fwd_hd: head_dim=%d is not built (head dims 16 and 24)", head_dim);
    auto f = head_dim == 16 ? attn_fwd<16> : attn_fwd<24>;
    return f(q, k, v, qkv_row_stride, bias, tok_off, graph_order, B, H, ntok, T, Tp, t_max_host, t_min_host, scale, drop_p, seed,
             seed_dev, out, lse, stream);
}

extern "C" int32_t mobgt_attn_fwd(const void *q, const void *k, const void *v, int64_t qkv_row_stride, const void *bias,
                                  const int32_t *tok_off, const int32_t *graph_order, int32_t B, int32_t H, int32_t ntok,
                                  int32_t T, int32_t Tp, int32_t t_max_host, int32_t t_min_host, float scale, float drop_p, uint64_t seed,
                                  const void *seed_dev, void *out, float *lse, void *stream) {
    return mobgt_attn_fwd_hd(q, k, v, qkv_row_stride, bias, tok_off, graph_order, B, H, ntok, T, Tp, t_max_host, t_min_host, scale,
                             drop_p, seed, seed_dev, out, lse, 24, stream);
}
