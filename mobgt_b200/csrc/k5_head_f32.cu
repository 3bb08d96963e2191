// K5 in fp32 mode — POI-logit head in IEEE fp32 on the CUDA cores, fused with the same per-row top-k and rank epilogue as
// K5 (csrc/k5_head.cu).  `--precision 32` evaluates with it: the reference ranks fp32 logits (model_fqandtoyo.py:48-131,
// 1530-1597), and bf16-rounded operands move most target ranks of a 60 000-POI head.
//
// Arithmetic (one fixed order per logit, whatever the tiling, the split count or the vocabulary shard):
//     s = 0;  for k = 0 .. K-1 ascending:  s = fmaf(z[row][k], W[col][k], s);      logit = bias ? s + bias[col] : s
// Every fmaf and the final add are single IEEE roundings (__fmaf_rn / __fadd_rn); no tensor-core instruction is used.  Mode 0
// (the target's own logit) runs the same chain, so the target's logit compares equal to st and never counts against itself.
//
// mode 1 (k5_head_f32_kernel) — one CTA of 256 threads per (64-row tile of z, vocabulary split):
//   * the z tile stays resident in shared memory, [64][K + 4] f32 (83 KB at K = 320);
//   * W streams through a double-buffered ring of [128 vocabulary rows][32 K-columns] chunks (cp.async, zero-filled past V);
//   * thread (ty, tx) = (tid / 16, tid % 16) owns a 4 x 8 register micro-tile: rows ty + 16 i, columns tx + 16 j; one K-step
//     of 4 reads 4 + 8 float4 words of shared memory for 128 FFMAs;
//   * after each 128-column tile the logits (+ bias) go to a [64][132] shared tile; thread (r, q) = (tid / 4, tid % 4) then
//     scans columns q, q + 4, ... of row r in ascending order: #(s > s_t), #(s == s_t and col < t), and a register-resident
//     sorted top-k list (64-bit keys: order-preserving value bits | ~global index, so ties go to the lower index).
//   Each (row, split, q) emits one list + its two counts: nsplit = 4 x (vocabulary splits), merged by mobgt_topk_merge.
// mode 0 (k5_target_logit_f32_kernel) — one thread per row runs the fmaf chain of its target's column.
#include "common.cuh"

namespace mobgt {
namespace headf32 {

constexpr int kBM = 64;                // z rows per CTA
constexpr int kBN = 128;               // vocabulary rows (logit columns) per tile
constexpr int kKC = 32;                // K-columns per W chunk
constexpr int kWP = kKC + 4;           // W chunk pitch (floats): 16 consecutive vocabulary rows hit distinct bank quads
constexpr int kLP = kBN + 4;           // logit tile pitch (floats): the 32 (r, q) readers of a column step hit 32 banks
constexpr int kThreads = 256;
constexpr int kListsPerCta = 4;        // scanner threads per row
constexpr int kMaxK = 320;
constexpr int kMaxTop = 32;

struct Params {
    const float *z, *W, *bias;
    const int32_t *target;
    float *st;
    float *topk_val;        // [M, nsplit, k]
    int32_t *topk_idx;      // [M, nsplit, k]
    int32_t *cnt_gt, *cnt_eq;   // [M, nsplit]
    float *logits;          // optional [M, V]
    int M, V, K, k, nsplit;
    int64_t vocab_offset;
};

__device__ __forceinline__ uint32_t f2ord(float v) {
    const uint32_t u = __float_as_uint(v);
    return u ^ ((uint32_t)((int32_t)u >> 31) | 0x80000000u);
}
__device__ __forceinline__ float ord2f(uint32_t o) {
    return __uint_as_float((o & 0x80000000u) ? (o ^ 0x80000000u) : ~o);
}

__device__ __forceinline__ void cp_async16(uint32_t dst, const void *src, bool valid) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(valid ? 16 : 0) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait1() { asm volatile("cp.async.wait_group 1;" ::: "memory"); }

template <int LK>
__device__ __forceinline__ void list_insert(unsigned long long (&list)[LK], unsigned long long key) {
    list[LK - 1] = key;      // precondition: key > list[LK-1]
#pragma unroll
    for (int j = LK - 1; j > 0; --j) {
        const unsigned long long a = list[j - 1], b = list[j];
        const bool sw = b > a;
        list[j - 1] = sw ? b : a;
        list[j] = sw ? a : b;
    }
}

template <int LK>
__global__ void __launch_bounds__(kThreads, 1) k5_head_f32_kernel(const Params p) {
    extern __shared__ __align__(16) float smem[];
    const int K = p.K;
    const int zp = K + 4;
    float *sZ = smem;                                  // [kBM][K + 4]
    float *sW = sZ + kBM * zp;                         // [2][kBN][kWP]
    float *sL = sW + 2 * kBN * kWP;                    // [kBM][kLP]

    const int tid = threadIdx.x;
    const int ty = tid >> 4, tx = tid & 15;
    const int m0 = blockIdx.x * kBM;
    const int ntiles = ceil_div(p.V, kBN);
    const int tps = ceil_div(ntiles, (int)gridDim.y);
    const int n_begin = blockIdx.y * tps, n_end = min(ntiles, n_begin + tps);
    const int T = max(0, n_end - n_begin);
    const int nch = ceil_div(K, kKC);

    // W chunk g = (tile g / nch, K-columns (g % nch) * 32 ...): 128 rows x 8 float4 words, 4 per thread
    auto load_chunk = [&](int g, int buf) {
        const int n = n_begin + g / nch, k0 = (g % nch) * kKC;
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int e = tid + u * kThreads;
            const int rr = e >> 3, c4 = (e & 7) * 4;
            const int col = n * kBN + rr;
            const bool ok = col < p.V && k0 + c4 < K;
            const float *src = p.W + (ok ? (size_t)col * K + k0 + c4 : 0);
            cp_async16((uint32_t)__cvta_generic_to_shared(sW + ((size_t)buf * kBN + rr) * kWP + c4), src, ok);
        }
    };

    if (T > 0) load_chunk(0, 0);
    cp_async_commit();
    // the z tile, resident for the whole CTA (rows past M read as 0 and are never reported)
    for (int e = tid; e < kBM * (K / 4); e += kThreads) {
        const int r = e / (K / 4), c4 = (e % (K / 4)) * 4;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (m0 + r < p.M) v = __ldg(reinterpret_cast<const float4 *>(p.z + (size_t)(m0 + r) * K + c4));
        *reinterpret_cast<float4 *>(sZ + r * zp + c4) = v;
    }

    // scanner state: row r, columns q (mod 4) of every tile
    const int r = tid >> 2, q = tid & 3;
    const int row = m0 + r;
    const bool row_ok = row < p.M;
    const long long tgt = row_ok ? (long long)p.target[row] : -1;
    const long long tl64 = tgt < 0 ? -1 : tgt - p.vocab_offset;       // target column inside this shard (any sign / size)
    const int tloc = tl64 < 0 ? -1 : (tl64 > 0x7fffff00ll ? 0x7fffff00 : (int)tl64);
    const float st = row_ok ? p.st[row] : 0.f;
    unsigned long long list[LK];
#pragma unroll
    for (int j = 0; j < LK; ++j) list[j] = 0ull;
    float thr = -INFINITY;        // value of list[LK-1] once the list is full
    int cgt = 0, ceq = 0;

    float acc[4][8];
    for (int g = 0; g < T * nch; ++g) {
        const int c = g % nch;
        if (c == 0) {
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;
        }
        if (g + 1 < T * nch) load_chunk(g + 1, (g + 1) & 1);
        cp_async_commit();
        cp_async_wait1();
        __syncthreads();
        const float *w = sW + (size_t)(g & 1) * kBN * kWP + tx * kWP;
        const float *zr = sZ + ty * zp + c * kKC;
        const int nq = min(kKC, K - c * kKC) / 4;
#pragma unroll
        for (int kq = 0; kq < kKC / 4; ++kq) {
            if (kq < nq) {
                float4 a[4];
#pragma unroll
                for (int i = 0; i < 4; ++i) a[i] = *reinterpret_cast<const float4 *>(zr + i * 16 * zp + kq * 4);
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const float4 b = *reinterpret_cast<const float4 *>(w + j * 16 * kWP + kq * 4);
#pragma unroll
                    for (int i = 0; i < 4; ++i) {          // k ascending inside every accumulator
                        acc[i][j] = __fmaf_rn(a[i].x, b.x, acc[i][j]);
                        acc[i][j] = __fmaf_rn(a[i].y, b.y, acc[i][j]);
                        acc[i][j] = __fmaf_rn(a[i].z, b.z, acc[i][j]);
                        acc[i][j] = __fmaf_rn(a[i].w, b.w, acc[i][j]);
                    }
                }
            }
        }
        __syncthreads();          // the buffer is refilled by the next iteration's prefetch
        if (c != nch - 1) continue;

        // ---- tile finished: logits (+ bias) to shared memory, then the per-row scan
        const int cb = (n_begin + g / nch) * kBN;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const int col = cb + tx + 16 * j;
            const bool cok = col < p.V;
            const float b = (p.bias && cok) ? __ldg(p.bias + col) : 0.f;
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const float v = p.bias ? __fadd_rn(acc[i][j], b) : acc[i][j];
                sL[(ty + 16 * i) * kLP + tx + 16 * j] = v;
                if (p.logits != nullptr && cok && m0 + ty + 16 * i < p.M) p.logits[(size_t)(m0 + ty + 16 * i) * p.V + col] = v;
            }
        }
        __syncthreads();
        const int ncol = min(kBN, p.V - cb);
        const float *lr = sL + r * kLP;
#pragma unroll 4
        for (int cc = q; cc < ncol; cc += 4) {
            const float v = lr[cc];
            const int col = cb + cc;
            cgt += (int)(v > st);
            ceq += (int)((v == st) & (col < tloc));
            if (v >= thr) {          // columns arrive in ascending order: an equal value only wins a tie inside the key
                const uint32_t gi = (uint32_t)(p.vocab_offset + col);
                const unsigned long long key = ((unsigned long long)f2ord(v) << 32) | (uint32_t)(~gi);
                if (key > list[LK - 1]) {
                    list_insert<LK>(list, key);
                    if (list[LK - 1] != 0ull) thr = ord2f((uint32_t)(list[LK - 1] >> 32));
                }
            }
        }
        // sL is rewritten only after the next tile's chunk loop, which passes two __syncthreads()
    }

    if (row_ok) {
        const size_t o = (size_t)row * p.nsplit + (size_t)blockIdx.y * kListsPerCta + q;
#pragma unroll
        for (int j = 0; j < LK; ++j) {
            if (j < p.k) {
                const unsigned long long key = list[j];
                p.topk_val[o * p.k + j] = key ? ord2f((uint32_t)(key >> 32)) : -INFINITY;
                p.topk_idx[o * p.k + j] = key ? (int32_t)(~(uint32_t)key) : -1;
            }
        }
        p.cnt_gt[o] = cgt;
        p.cnt_eq[o] = ceq;
    }
}

// mode 0: st[row] = logit of the row's target, through the same fmaf chain, for the rows whose target lies in this shard
__global__ void __launch_bounds__(128) k5_target_logit_f32_kernel(const Params p) {
    const int row = blockIdx.x * blockDim.x + threadIdx.x;
    if (row >= p.M) return;
    const long long t = (long long)p.target[row] - p.vocab_offset;
    if (p.target[row] < 0 || t < 0 || t >= p.V) return;
    const float4 *zr = reinterpret_cast<const float4 *>(p.z + (size_t)row * p.K);
    const float4 *wr = reinterpret_cast<const float4 *>(p.W + (size_t)t * p.K);
    float s = 0.f;
    for (int k4 = 0; k4 < p.K / 4; ++k4) {
        const float4 a = __ldg(zr + k4), b = __ldg(wr + k4);
        s = __fmaf_rn(a.x, b.x, s);
        s = __fmaf_rn(a.y, b.y, s);
        s = __fmaf_rn(a.z, b.z, s);
        s = __fmaf_rn(a.w, b.w, s);
    }
    p.st[row] = p.bias ? __fadd_rn(s, __ldg(p.bias + t)) : s;
}

}  // namespace headf32
}  // namespace mobgt

using namespace mobgt;

extern "C" int32_t mobgt_head_topk_f32(const float *z, const float *W, const float *bias, const int32_t *target, int32_t M,
                                       int32_t V, int32_t K, int64_t vocab_offset, int32_t k, int32_t nsplit, int32_t mode,
                                       float *st, float *topk_val, int32_t *topk_idx, int32_t *cnt_gt, int32_t *cnt_eq,
                                       float *logits_dump, void *thr_share, void *stream) {
    using namespace headf32;
    (void)thr_share;
    MOBGT_REQUIRE(z && W && target && st, MOBGT_ERR_NULL, "mobgt_head_topk_f32: null pointer");
    MOBGT_REQUIRE(mode == 0 || mode == 1, MOBGT_ERR_BAD_SHAPE, "mobgt_head_topk_f32: mode=%d must be 0 or 1", mode);
    MOBGT_REQUIRE(mode == 0 || (topk_val && topk_idx && cnt_gt && cnt_eq), MOBGT_ERR_NULL, "mobgt_head_topk_f32: null output");
    MOBGT_REQUIRE(K % 4 == 0 && K >= 4 && K <= kMaxK, MOBGT_ERR_BAD_SHAPE,
                  "mobgt_head_topk_f32: K=%d must be a multiple of 4 in [4, 320]", K);
    MOBGT_REQUIRE(k >= 1 && k <= kMaxTop, MOBGT_ERR_BAD_SHAPE, "mobgt_head_topk_f32: k=%d must be in [1, 32]", k);
    MOBGT_REQUIRE(mode == 0 || (nsplit >= 4 && nsplit <= 160 && nsplit % 4 == 0), MOBGT_ERR_BAD_SHAPE,
                  "mobgt_head_topk_f32: nsplit=%d must be a multiple of 4 in [4, 160] (four lists per vocabulary split)", nsplit);
    MOBGT_REQUIRE(((uintptr_t)z & 15) == 0 && ((uintptr_t)W & 15) == 0, MOBGT_ERR_BAD_SHAPE,
                  "mobgt_head_topk_f32: z and W must be 16-byte aligned");
    MOBGT_REQUIRE(M >= 0 && V >= 0, MOBGT_ERR_BAD_SHAPE, "mobgt_head_topk_f32: M=%d V=%d", M, V);
    if (M == 0 || V == 0) return MOBGT_OK;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    Params p{z, W, bias, target, st, topk_val, topk_idx, cnt_gt, cnt_eq, logits_dump, M, V, K, k, nsplit, vocab_offset};
    if (mode == 0) {
        k5_target_logit_f32_kernel<<<ceil_div(M, 128), 128, 0, s>>>(p);
        MOBGT_LAUNCH_OK("k5_target_logit_f32_kernel");
        return MOBGT_OK;
    }
    const size_t smem = ((size_t)kBM * (K + 4) + (size_t)2 * kBN * kWP + (size_t)kBM * kLP) * sizeof(float);
    const dim3 grid((unsigned)ceil_div(M, kBM), (unsigned)(nsplit / kListsPerCta));
    auto launch = [&](auto kern) -> int32_t {
        MOBGT_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        kern<<<grid, kThreads, smem, s>>>(p);
        return MOBGT_OK;
    };
    // the list length is a compile-time constant (register-resident list): the smallest built size >= k
    const int32_t rc = k <= 10 ? launch(k5_head_f32_kernel<10>) : k <= 20 ? launch(k5_head_f32_kernel<20>) : launch(k5_head_f32_kernel<32>);
    if (rc) return rc;
    MOBGT_LAUNCH_OK("k5_head_f32_kernel");
    return MOBGT_OK;
}
