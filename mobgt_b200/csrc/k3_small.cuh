// Interface between the attention entry points (k3_attn_fwd.cu / k3_attn_bwd.cu) and the small-graph SIMT kernels
// (k3_attn_small.cu).
#pragma once
#include <cuda_bf16.h>

#include "common.cuh"

namespace mobgt {

constexpr int kSmallT = 16;   // graphs of at most this many tokens (n + 1) take the SIMT path (9 trajectory graphs in 10)

// Head-dim dependent shapes of the tensor-core kernels (k3_attn_fwd.cu / k3_attn_bwd.cu).  An operand box is the no-swizzle
// [chunk][128 rows][16 B] image of umma.cuh; along d the MMA K (S, dP) and N (O, dV, dK, dQ) extent is d rounded up to 16:
// d = 24 -> 32 (three data chunks + one zero chunk), d = 16 -> 16 (two data chunks, no padding).
template <int kD>
struct AttnShape {
    static_assert(kD == 16 || kD == 24, "the attention kernels are built for head dims 16 and 24");
    static constexpr int kChunks = kD / 8;                 // 16-byte chunks of data per row (the TMA box depth)
    static constexpr int kDPad = (kD + 15) / 16 * 16;      // MMA extent along d
    static constexpr int kBoxBytes = (kDPad / 8) * 128 * 16;
    static constexpr int kBoxTxBytes = kChunks * 128 * 16;
    static constexpr int kSegs = 240 / kD;                 // single-token tail mat-vecs: 240 threads = (segment, element)
};

// 8 kC bf16 (kC 16-byte words) -> fp32
template <int kC>
__device__ __forceinline__ void unpack_words(const uint4 (&w)[kC], float (&f)[8 * kC]) {
#pragma unroll
    for (int c = 0; c < kC; ++c) {
        const uint32_t u[4] = {w[c].x, w[c].y, w[c].z, w[c].w};
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            f[8 * c + 2 * e] = __uint_as_float(u[e] << 16);
            f[8 * c + 2 * e + 1] = __uint_as_float(u[e] & 0xFFFF0000u);
        }
    }
}

struct SmallAttnParams {
    const int32_t *tok_off;
    const int32_t *order;             // [B] graph ids in launch order (descending size) or NULL
    const __nv_bfloat16 *q, *k, *v;   // [ntok, qkv_stride]
    int64_t qkv_stride;
    const __nv_bfloat16 *bias;        // [B,H,T,Tp]
    int H, T, Tp;
    float scale;
    int small_t;                      // graphs with more tokens are left to the tensor-core kernels
    AttnDrop drop;
    // forward
    __nv_bfloat16 *out;               // [ntok, H*d]
    float *lse;                       // [ntok, H]   (backward: input)
    // backward
    const __nv_bfloat16 *o, *dout;    // [ntok, H*d]
    __nv_bfloat16 *dq, *dk, *dv;      // [ntok, dqkv_stride]
    int64_t dqkv_stride;
    void *dbias;                      // f32 (accumulate 0 / 1) or bf16 (accumulate 2) [B,H,T,Tp]
    int accumulate;
};

// H % 4 == 0; kD: head dim 16 or 24 (explicitly instantiated in k3_attn_small.cu)
template <int kD> int32_t launch_small_attn_fwd(const SmallAttnParams &p, int B, cudaStream_t s);
template <int kD> int32_t launch_small_attn_bwd(const SmallAttnParams &p, int B, cudaStream_t s);

// Graphs of more than kLargeT tokens (up to MOBGT_MAX_MODEL_NODES + 1) are computed by the SIMT kernels of k3_attn_large.cu;
// the tensor-core kernels skip them on the device and size their shared memory for at most kLargeT tokens.
constexpr int kLargeT = MOBGT_MAX_NODES + 1;

struct LargeAttnParams {
    const int32_t *tok_off;
    const int32_t *order;             // [B] graph ids in launch order or NULL
    const void *q, *k, *v;            // TE [ntok, qkv_stride]
    int64_t qkv_stride;
    const void *bias;                 // TE [B,H,T,Tp]
    int H, T, Tp;
    float scale;
    int t_lo;                         // graphs of more than t_lo tokens belong to these kernels
    AttnDrop drop;
    void *out;                        // TE [ntok, H*d]
    float *lse;                       // [ntok, H]   (backward: input)
    const void *o, *dout;             // TE [ntok, H*d]
    void *dq, *dk, *dv;               // TE [ntok, dqkv_stride]
    int64_t dqkv_stride;
    void *dbias;                      // f32 (accumulate 0 / 1) or bf16 (accumulate 2) [B,H,T,Tp]
    int accumulate;
};

// TE: __nv_bfloat16 (forward and backward) or float (backward); kD: 16 or 24; t_max: the largest token count of the batch.
// Explicitly instantiated in k3_attn_large.cu.
template <typename TE, int kD> int32_t launch_large_attn_fwd(const LargeAttnParams &p, int B, int t_max, cudaStream_t s);
template <typename TE, int kD> int32_t launch_large_attn_bwd(const LargeAttnParams &p, int B, int t_max, cudaStream_t s);

}  // namespace mobgt
