// K1 — batched all-pairs shortest paths + path-edge extraction (sm_100a).
//
// Replaces the reference's Cython preprocessing, bit-exactly:
//   algos.floyd_warshall   /root/reference/graphormer/algos.pyx:9-54
//   algos.get_all_edges    algos.pyx:57-62
//   algos.gen_edge_input   algos.pyx:65-96
// as driven by preprocess_item (wrapper.py:42-61,99) and sliced by the collators
// (collator.py:323).
//
// Design (see DESIGN.md §K1):
//   * one thread-block CLUSTER per graph; the cluster's C CTAs (C = 1,2,4,8) each own a
//     slice of W columns of the n x n state, kept in shared memory as packed uint16
//     (M = distance, X = next-hop; optionally P = the reference's `path` matrix);
//   * Floyd-Warshall runs k strictly ascending (the reference's relaxation order decides
//     `path`, algos.pyx:35-45); inside one k the n*n relaxations are order-free because row k
//     and column k are fixed points of step k (M[k][k] == 0, strict '>');
//     column k of M and X is broadcast to every CTA through distributed shared memory by the
//     thread that just relaxed it, so a step costs ONE (cluster) barrier;
//   * 8 cells per 128-bit shared-memory access, 2 cells per ALU op (__vminu2/__vcmpltu2);
//   * the reference's recursive in-order expansion get_all_edges(i,j) is replaced by the
//     next-hop matrix X maintained inside FW:  X[i][j] = j initially, X[i][j] = X[i][k] on a
//     strict improvement through k != 0 (k == 0 leaves X alone: this reproduces the reference's
//     "path == 0 means direct" short-circuit, algos.pyx:59-60).  DESIGN.md proves that
//     walking cur = X[cur][j] emits exactly the reference's hop sequence;
//   * the walk writes only the first `hops` hop slots (collator.py:323 slices the rest away),
//     staged per warp in shared memory and stored as coalesced 32-bit words;
//   * graphs of 513..1024 nodes (the algos drop-in only) use k1_apsp_large_kernel: M alone in the
//     shared memory of an 8- or 16-CTA cluster, `path` in global memory, expanded by
//     k1_walk_from_path_kernel in the same call.
#include <cooperative_groups.h>
#include <cstdlib>

#include "common.cuh"

namespace cg = cooperative_groups;

namespace mobgt {

struct K1Params {
    const uint8_t *feat;
    const int32_t *n;
    const int64_t *sq_off;
    const int32_t *gids;
    int hops;   // byte stride of one edge_in row (multiple of 4)
    int dk;     // hop slots actually walked: multi_hop_max_dist (collator.py:323); slots [dk, hops) stay "no hop"
    int shift;
    int16_t *dist;
    int16_t *path;
    uint8_t *edge_in;
    int32_t *maxdist;
};

constexpr uint32_t kInf = MOBGT_UNREACHABLE;
constexpr uint16_t kNoWalk = 0x8000u;   // flag bit on X[i][j]: no walk STARTS at (i,j); the low bits stay a valid next hop

__device__ __forceinline__ uint32_t pick16(const uint4 &v, int e) {
    const int w = e >> 1;
    const uint32_t x = (w == 0) ? v.x : (w == 1) ? v.y : (w == 2) ? v.z : v.w;
    return (e & 1) ? (x >> 16) : (x & 0xFFFFu);
}

// one packed relaxation of 2 cells: m = min(m, rk + mik2) per half-word in ONE instruction (VIADDMNMX.U16x2; the halves are
// <= 1020, no carry across the half-word boundary); returns old ^ new — a half-word is non-zero iff that cell STRICTLY improved
// (algos.pyx:41 `>`).  The full 0xFFFF / 0 select masks are only built on the rare path (half_masks): the packed compare
// __vcmpltu2 is emulated with six instructions per word on sm_100 and used to be 60 % of the inner loop.
__device__ __forceinline__ uint32_t relax2(uint32_t &m, uint32_t rk, uint32_t mik2) {
    const uint32_t nm = __viaddmin_u16x2(rk, mik2, m);
    const uint32_t diff = nm ^ m;
    m = nm;
    return diff;
}
__device__ __forceinline__ uint32_t half_masks(uint32_t diff) {
    return ((diff & 0xFFFFu) ? 0xFFFFu : 0u) | ((diff >> 16) ? 0xFFFF0000u : 0u);
}

__host__ __device__ inline int k1_W(int n, int C) { return round_up(ceil_div(n, C), 8); }

__host__ inline size_t k1_smem_bytes(int n, int C, bool with_path, int nthreads, int hops, bool with_feat) {
    const int W = k1_W(n, C);
    const int n8 = round_up(n, 8);
    size_t b = (size_t)n * W * 2 * (with_path ? 3 : 2);
    b += (size_t)4 * n8 * 2;                       // colM[2][n8], colX[2][n8]
    b += (size_t)(nthreads / 32) * 32 * hops;      // per-warp walk staging
    b = (b + 15) / 16 * 16;
    if (with_feat) b += (size_t)round_up(n * n, 16);   // the graph's edge-feature bytes for the walk
    return b + 16;
}

template <bool WITH_PATH>
__global__ void __launch_bounds__(1024) k1_apsp_kernel(const K1Params p, const int C, const int feat_in_smem) {
    cg::cluster_group cluster = cg::this_cluster();
    const int crank = (C > 1) ? (int)cluster.block_rank() : 0;
    const int gl = blockIdx.x / C;
    const int g = p.gids ? p.gids[gl] : gl;
    const int n = p.n[g];
    const int64_t off = p.sq_off[g];
    const int W = k1_W(n, C);
    const int c0 = crank * W;
    const int wc = max(0, min(W, n - c0));  // valid columns owned by this CTA
    const int n8 = round_up(n, 8);
    const int cpr = W >> 3;  // 8-cell chunks per row
    const int tid = threadIdx.x, NT = blockDim.x;

    extern __shared__ __align__(16) uint8_t smem_raw[];
    uint16_t *Msh = reinterpret_cast<uint16_t *>(smem_raw);
    uint16_t *Xsh = Msh + (size_t)n * W;
    uint16_t *Psh = Xsh + (size_t)n * W;
    uint16_t *colM = WITH_PATH ? (Psh + (size_t)n * W) : Psh;  // [2][n8]
    uint16_t *colX = colM + 2 * n8;                             // [2][n8]
    uint8_t *stage = reinterpret_cast<uint8_t *>(colX + 2 * n8);
    // the walk reads one edge-feature byte per hop at a data-dependent address: a chain of up to `dk` dependent loads per pair.
    // With the n x n bytes of the graph staged in shared memory each link of the chain is an LDS (~30 cycles) instead of a
    // global load (several hundred); the launch provisions the space whenever it fits next to the Floyd-Warshall state.
    uint8_t *featS = nullptr;
    if (feat_in_smem) {
        const size_t so = (((size_t)(stage - smem_raw) + (size_t)(blockDim.x / 32) * 32 * p.hops) + 15) / 16 * 16;
        featS = smem_raw + so;
    }

    const uint8_t *feat = p.feat + off;
    const int ntask = n * cpr;
    if (featS != nullptr) {
        const int nb = n * n;
        if (((uintptr_t)feat & 15) == 0) {
            for (int t = tid; t < (nb >> 4); t += NT) reinterpret_cast<uint4 *>(featS)[t] = __ldg(reinterpret_cast<const uint4 *>(feat) + t);
            for (int t = (nb & ~15) + tid; t < nb; t += NT) featS[t] = __ldg(feat + t);
        } else {
            for (int t = tid; t < nb; t += NT) featS[t] = __ldg(feat + t);
        }
    }

    // ---- init (algos.pyx:27-32): diag 0, edge 1, else 510; X[i][j] = j; P = 0 ----------------
    for (int t = tid; t < ntask; t += NT) {
        const int i = t / cpr, q = t - i * cpr;
        uint32_t mw[4], xw[4];
#pragma unroll
        for (int e2 = 0; e2 < 4; ++e2) {
            uint32_t mm[2], xx[2];
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const int j = c0 + q * 8 + e2 * 2 + h;
                uint32_t m = kInf;
                if (j < n) {
                    const uint8_t f = __ldg(feat + (size_t)i * n + j);
                    m = (i == j) ? 0u : (f ? 1u : kInf);
                }
                mm[h] = m;
                xx[h] = (uint32_t)j & 0xFFFFu;
            }
            mw[e2] = mm[0] | (mm[1] << 16);
            xw[e2] = xx[0] | (xx[1] << 16);
        }
        *reinterpret_cast<uint4 *>(Msh + (size_t)i * W + q * 8) = make_uint4(mw[0], mw[1], mw[2], mw[3]);
        *reinterpret_cast<uint4 *>(Xsh + (size_t)i * W + q * 8) = make_uint4(xw[0], xw[1], xw[2], xw[3]);
        if (WITH_PATH) *reinterpret_cast<uint4 *>(Psh + (size_t)i * W + q * 8) = make_uint4(0, 0, 0, 0);
    }
    // column 0 of M and X for step k = 0: every CTA derives it from the input itself
    for (int i = tid; i < n; i += NT) {
        const uint8_t f = __ldg(feat + (size_t)i * n);
        colM[i] = (uint16_t)((i == 0) ? 0u : (f ? 1u : kInf));
        colX[i] = 0;
    }
    if (C > 1) cluster.sync(); else __syncthreads();

    // ---- Floyd-Warshall, k strictly ascending (algos.pyx:35-45) ---------------------------------
    const int dr = NT / cpr, dq = NT - dr * cpr;
    const int i0 = tid / cpr, q0 = tid - i0 * cpr;
    for (int k = 0; k < n; ++k) {
        const uint16_t *cM = colM + (k & 1) * n8;
        const uint16_t *cX = colX + (k & 1) * n8;
        const int nb = ((k + 1) & 1) * n8;
        const int kn = k + 1;
        const bool own_next = (kn < n) && (kn >= c0) && (kn < c0 + W);
        const int qn = own_next ? ((kn - c0) >> 3) : -1;
        const int en = (kn - c0) & 7;
        const uint32_t k2 = (uint32_t)k * 0x10001u;
        const uint16_t *rowk = Msh + (size_t)k * W;

        int i = i0, q = q0;
        for (int t = tid; t < ntask; t += NT) {
            const uint32_t mik = cM[i];
            const bool pub = (q == qn);
            if (mik < kInf || pub) {
                uint16_t *mp = Msh + (size_t)i * W + q * 8;
                uint16_t *xp = Xsh + (size_t)i * W + q * 8;
                uint4 m4 = *reinterpret_cast<const uint4 *>(mp);
                uint4 x4;
                bool have_x = false;
                if (mik < kInf) {
                    const uint4 r4 = *reinterpret_cast<const uint4 *>(rowk + q * 8);
                    const uint32_t mik2 = mik * 0x10001u;
                    const uint32_t d0 = relax2(m4.x, r4.x, mik2);
                    const uint32_t d1 = relax2(m4.y, r4.y, mik2);
                    const uint32_t d2 = relax2(m4.z, r4.z, mik2);
                    const uint32_t d3 = relax2(m4.w, r4.w, mik2);
                    if (d0 | d1 | d2 | d3) {
                        *reinterpret_cast<uint4 *>(mp) = m4;
                        if (k != 0) {  // k == 0: path stays 0 == "direct" (algos.pyx:59-60) -> X untouched
                            const uint32_t l0 = half_masks(d0), l1 = half_masks(d1), l2 = half_masks(d2), l3 = half_masks(d3);
                            x4 = *reinterpret_cast<const uint4 *>(xp);
                            const uint32_t xik2 = (uint32_t)cX[i] * 0x10001u;
                            x4.x = (x4.x & ~l0) | (xik2 & l0);
                            x4.y = (x4.y & ~l1) | (xik2 & l1);
                            x4.z = (x4.z & ~l2) | (xik2 & l2);
                            x4.w = (x4.w & ~l3) | (xik2 & l3);
                            *reinterpret_cast<uint4 *>(xp) = x4;
                            have_x = true;
                            if (WITH_PATH) {
                                uint16_t *pp = Psh + (size_t)i * W + q * 8;
                                uint4 p4 = *reinterpret_cast<const uint4 *>(pp);
                                p4.x = (p4.x & ~l0) | (k2 & l0);
                                p4.y = (p4.y & ~l1) | (k2 & l1);
                                p4.z = (p4.z & ~l2) | (k2 & l2);
                                p4.w = (p4.w & ~l3) | (k2 & l3);
                                *reinterpret_cast<uint4 *>(pp) = p4;
                            }
                        }
                    }
                }
                if (pub) {  // broadcast column k+1 (post-step-k values) to every CTA of the cluster
                    if (!have_x) x4 = *reinterpret_cast<const uint4 *>(xp);
                    const uint16_t mv = (uint16_t)pick16(m4, en);
                    const uint16_t xv = (uint16_t)pick16(x4, en);
                    if (C > 1) {
                        for (int r = 0; r < C; ++r) {
                            cluster.map_shared_rank(colM, r)[nb + i] = mv;
                            cluster.map_shared_rank(colX, r)[nb + i] = xv;
                        }
                    } else {
                        colM[nb + i] = mv;
                        colX[nb + i] = xv;
                    }
                }
            }
            q += dq;
            i += dr;
            if (q >= cpr) { q -= cpr; ++i; }
        }
        if (C > 1) cluster.sync(); else __syncthreads();
    }

    // ---- finalize (algos.pyx:48-52) + dist / path / maxdist outputs -----------------------------
    int local_max = 0;
    for (int t = tid; t < ntask; t += NT) {
        const int i = t / cpr, q = t - i * cpr;
        const uint4 m4 = *reinterpret_cast<const uint4 *>(Msh + (size_t)i * W + q * 8);
        uint4 x4 = *reinterpret_cast<const uint4 *>(Xsh + (size_t)i * W + q * 8);
        uint4 p4 = make_uint4(0, 0, 0, 0);
        if (WITH_PATH) p4 = *reinterpret_cast<const uint4 *>(Psh + (size_t)i * W + q * 8);
        uint32_t xo[4] = {x4.x, x4.y, x4.z, x4.w};
#pragma unroll
        for (int e = 0; e < 8; ++e) {
            const int j = c0 + q * 8 + e;
            const uint32_t m = pick16(m4, e);
            const bool unreach = (m >= kInf) || (j >= n);
            // the reference skips a pair when path == 510 (algos.pyx:87-88); for n > 510 that also hits REACHABLE
            // pairs whose last improving intermediate is node 510 -- reproduced here (P is kept whenever n > 510)
            const bool skip510 = WITH_PATH && (pick16(p4, e) == kInf);
            if (unreach || i == j || skip510) {
                // flag only: walks of OTHER pairs (i',j) that pass through i still need X[i][j] (a skip510 pair is reachable)
                xo[e >> 1] |= (e & 1) ? ((uint32_t)kNoWalk << 16) : (uint32_t)kNoWalk;
            }
            if (j < n) {
                const size_t o = (size_t)off + (size_t)i * n + j;
                p.dist[o] = (int16_t)(m + p.shift);
                if (WITH_PATH && p.path != nullptr) p.path[o] = (int16_t)(unreach ? kInf : pick16(p4, e));
                local_max = max(local_max, (int)m);
            }
        }
        *reinterpret_cast<uint4 *>(Xsh + (size_t)i * W + q * 8) = make_uint4(xo[0], xo[1], xo[2], xo[3]);
    }
#pragma unroll
    for (int s = 16; s > 0; s >>= 1) local_max = max(local_max, __shfl_xor_sync(0xffffffffu, local_max, s));
    if ((tid & 31) == 0 && ntask > 0) atomicMax(p.maxdist + g, local_max);
    __syncthreads();

    // ---- walk: first `hops` hops of the reference's in-order expansion (algos.pyx:85-94) -----
    if (p.edge_in != nullptr && wc > 0) {
        const int hops = p.hops;
        const int lane = tid & 31, warp = tid >> 5, nwarps = NT >> 5;
        uint8_t *st = stage + (size_t)warp * 32 * hops;
        const uint32_t none4 = (uint32_t)((p.shift - 1) & 0xFF) * 0x01010101u;
        const int hopw = hops >> 2;
        const int ngrp = ceil_div(wc, 32);
        const int nwt = n * ngrp;
        for (int wt = warp; wt < nwt; wt += nwarps) {
            const int i = wt / ngrp, cgp = wt - i * ngrp;
            const int jl = cgp * 32 + lane;
            const int j = c0 + jl;
            uint32_t *stw = reinterpret_cast<uint32_t *>(st) + lane * hopw;
            for (int w = 0; w < hopw; ++w) stw[w] = none4;
            if (jl < wc && !(Xsh[(size_t)i * W + jl] & kNoWalk)) {
                int cur = i;
                for (int h = 0; h < p.dk; ++h) {
                    const int nx = Xsh[(size_t)cur * W + jl] & (kNoWalk - 1);
                    const uint8_t f = featS ? featS[cur * n + nx] : __ldg(feat + (size_t)cur * n + nx);
                    st[lane * hops + h] = (uint8_t)(f + p.shift);
                    cur = nx;
                    if (cur == j) break;
                }
            }
            __syncwarp();
            const int npair = min(32, wc - cgp * 32);
            const int nwords = npair * hopw;
            uint32_t *dst = reinterpret_cast<uint32_t *>(p.edge_in + ((size_t)off + (size_t)i * n + c0 + cgp * 32) * hops);
            const uint32_t *src = reinterpret_cast<const uint32_t *>(st);
            for (int w = lane; w < nwords; w += 32) dst[w] = src[w];
            __syncwarp();
        }
    }
}

// ---- graphs of 513..1024 nodes (MOBGT_MAX_APSP_NODES) ------------------------------------------
// Same Floyd-Warshall (k strictly ascending, strict '>', saturating 510, one cluster barrier per k, column k of M broadcast
// through DSMEM), but only M stays in shared memory: the state of three matrices no longer fits a cluster at n = 600.  X is
// dropped and P, written only on a strict improvement, goes straight to the caller's `path` buffer: for n > 510 the
// reference's `path` is needed anyway (the skip510 rule reads it), and the walk then expands it with
// k1_walk_from_path_kernel, the reference's leftmost descent.  Rows of P start at any cell, so P is stored per cell.
constexpr int kLargeThreads = 1024;

__host__ inline size_t k1_large_smem_bytes(int n, int C) {
    return (size_t)n * k1_W(n, C) * 2 + (size_t)2 * round_up(n, 8) * 2 + 16;   // M slice + colM[2][n8]
}

__global__ void __launch_bounds__(kLargeThreads) k1_apsp_large_kernel(const K1Params p, const int C) {
    cg::cluster_group cluster = cg::this_cluster();
    const int crank = (int)cluster.block_rank();
    const int gl = blockIdx.x / C;
    const int g = p.gids ? p.gids[gl] : gl;
    const int n = p.n[g];
    const int64_t off = p.sq_off[g];
    const int W = k1_W(n, C);
    const int c0 = crank * W;
    const int n8 = round_up(n, 8);
    const int cpr = W >> 3;
    const int tid = threadIdx.x, NT = blockDim.x;

    extern __shared__ __align__(16) uint8_t smem_raw[];
    uint16_t *Msh = reinterpret_cast<uint16_t *>(smem_raw);
    uint16_t *colM = Msh + (size_t)n * W;   // [2][n8]
    const uint8_t *feat = p.feat + off;
    int16_t *P = p.path + off;
    const int ntask = n * cpr;

    // ---- init (algos.pyx:27-32): diag 0, edge 1, else 510; P = 0.  Cell (i, j) is owned by one thread for the whole kernel,
    // so its P stores (init, improvements, finalize) are ordered by program order alone.
    for (int t = tid; t < ntask; t += NT) {
        const int i = t / cpr, q = t - i * cpr;
        uint32_t mw[4];
#pragma unroll
        for (int e2 = 0; e2 < 4; ++e2) {
            uint32_t mm[2];
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const int j = c0 + q * 8 + e2 * 2 + h;
                uint32_t m = kInf;
                if (j < n) {
                    const uint8_t f = __ldg(feat + (size_t)i * n + j);
                    m = (i == j) ? 0u : (f ? 1u : kInf);
                    P[(size_t)i * n + j] = 0;
                }
                mm[h] = m;
            }
            mw[e2] = mm[0] | (mm[1] << 16);
        }
        *reinterpret_cast<uint4 *>(Msh + (size_t)i * W + q * 8) = make_uint4(mw[0], mw[1], mw[2], mw[3]);
    }
    for (int i = tid; i < n; i += NT) {
        const uint8_t f = __ldg(feat + (size_t)i * n);
        colM[i] = (uint16_t)((i == 0) ? 0u : (f ? 1u : kInf));
    }
    cluster.sync();

    // ---- Floyd-Warshall, k strictly ascending (algos.pyx:35-45) ---------------------------------
    const int dr = NT / cpr, dq = NT - dr * cpr;
    const int i0 = tid / cpr, q0 = tid - i0 * cpr;
    for (int k = 0; k < n; ++k) {
        const uint16_t *cM = colM + (k & 1) * n8;
        const int nb = ((k + 1) & 1) * n8;
        const int kn = k + 1;
        const bool own_next = (kn < n) && (kn >= c0) && (kn < c0 + W);
        const int qn = own_next ? ((kn - c0) >> 3) : -1;
        const int en = (kn - c0) & 7;
        const uint16_t *rowk = Msh + (size_t)k * W;

        int i = i0, q = q0;
        for (int t = tid; t < ntask; t += NT) {
            const uint32_t mik = cM[i];
            const bool pub = (q == qn);
            if (mik < kInf || pub) {
                uint16_t *mp = Msh + (size_t)i * W + q * 8;
                uint4 m4 = *reinterpret_cast<const uint4 *>(mp);
                if (mik < kInf) {
                    const uint4 r4 = *reinterpret_cast<const uint4 *>(rowk + q * 8);
                    const uint32_t mik2 = mik * 0x10001u;
                    const uint32_t d[4] = {relax2(m4.x, r4.x, mik2), relax2(m4.y, r4.y, mik2), relax2(m4.z, r4.z, mik2),
                                           relax2(m4.w, r4.w, mik2)};
                    if (d[0] | d[1] | d[2] | d[3]) {
                        *reinterpret_cast<uint4 *>(mp) = m4;
                        if (k != 0) {  // k == 0: path stays 0 == "direct" (algos.pyx:59-60)
                            const int jb = c0 + q * 8;
                            int16_t *pr = P + (size_t)i * n + jb;
#pragma unroll
                            for (int e = 0; e < 8; ++e)
                                if (((d[e >> 1] >> ((e & 1) * 16)) & 0xFFFFu) && jb + e < n) pr[e] = (int16_t)k;
                        }
                    }
                }
                if (pub) {  // broadcast column k+1 (post-step-k values) to every CTA of the cluster
                    const uint16_t mv = (uint16_t)pick16(m4, en);
                    for (int r = 0; r < C; ++r) cluster.map_shared_rank(colM, r)[nb + i] = mv;
                }
            }
            q += dq;
            i += dr;
            if (q >= cpr) { q -= cpr; ++i; }
        }
        cluster.sync();
    }

    // ---- finalize (algos.pyx:48-52) + dist / maxdist; unreachable pairs get path = 510 -------------
    int local_max = 0;
    for (int t = tid; t < ntask; t += NT) {
        const int i = t / cpr, q = t - i * cpr;
        const uint4 m4 = *reinterpret_cast<const uint4 *>(Msh + (size_t)i * W + q * 8);
#pragma unroll
        for (int e = 0; e < 8; ++e) {
            const int j = c0 + q * 8 + e;
            if (j < n) {
                const uint32_t m = pick16(m4, e);
                const size_t o = (size_t)i * n + j;
                p.dist[off + o] = (int16_t)(m + p.shift);
                if (m >= kInf) P[o] = (int16_t)kInf;
                local_max = max(local_max, (int)m);
            }
        }
    }
#pragma unroll
    for (int s = 16; s > 0; s >>= 1) local_max = max(local_max, __shfl_xor_sync(0xffffffffu, local_max, s));
    if ((tid & 31) == 0) atomicMax(p.maxdist + g, local_max);
}

// Stand-alone gen_edge_input from a floyd_warshall `path` matrix: hop h+1 of (cur -> j) is found
// by the leftmost descent of the reference's recursion (algos.pyx:57-62): t = j; while path[cur][t]
// != 0: t = path[cur][t].  One thread per ordered pair; walks the first `dk` hops and writes all `hops`
// slots of the row (the rest "no hop").  gids (may be NULL = identity) maps blockIdx.y to a graph.
// The API mirror, and the walk of the graphs above 512 nodes.
__global__ void k1_walk_from_path_kernel(const int16_t *__restrict__ path, const uint8_t *__restrict__ feat,
                                         const int32_t *__restrict__ n_arr, const int64_t *__restrict__ sq_off,
                                         const int32_t *__restrict__ gids, int hops, int dk, int shift,
                                         uint8_t *__restrict__ edge_in) {
    const int g = gids ? gids[blockIdx.y] : blockIdx.y;
    const int n = n_arr[g];
    const int64_t off = sq_off[g];
    const uint8_t none = (uint8_t)(shift - 1);
    for (int c = blockIdx.x * blockDim.x + threadIdx.x; c < n * n; c += gridDim.x * blockDim.x) {
        const int i = c / n, j = c - i * n;
        uint8_t *out = edge_in + ((size_t)off + c) * hops;
        int h = 0;
        const int pij = path[off + c];
        if (i != j && pij != (int)kInf) {
            int cur = i;
            for (; h < dk; ++h) {
                int t = j;
                for (int guard = 0; guard < n; ++guard) {
                    const int k = path[off + (size_t)cur * n + t];
                    if (k == 0) break;
                    t = k;
                }
                out[h] = (uint8_t)(feat[off + (size_t)cur * n + t] + shift);
                cur = t;
                if (cur == j) { ++h; break; }
            }
        }
        for (; h < hops; ++h) out[h] = none;
    }
}

// in_degree = row sums, out_degree = column sums of the bool adjacency (wrapper.py:97-98).
__global__ void k1_degree_kernel(const uint8_t *__restrict__ feat, const int32_t *__restrict__ n_arr,
                                 const int64_t *__restrict__ sq_off, const int64_t *__restrict__ node_off, int shift,
                                 int16_t *__restrict__ in_deg, int16_t *__restrict__ out_deg) {
    const int g = blockIdx.x;
    const int n = n_arr[g];
    const uint8_t *f = feat + sq_off[g];
    const int64_t no = node_off[g];
    for (int v = threadIdx.x; v < n; v += blockDim.x) {
        int r = 0, c = 0;
        for (int u = 0; u < n; ++u) {
            r += f[(size_t)v * n + u] != 0;
            c += f[(size_t)u * n + v] != 0;
        }
        in_deg[no + v] = (int16_t)(r + shift);
        out_deg[no + v] = (int16_t)(c + shift);
    }
}

// Threads per CTA: 8 tasks (8-cell chunks) per thread and k-step when the launch has enough graphs to fill the GPU with that
// (the preprocessing bench: thousands of graphs per launch); a launch of few graphs (one training batch of 256) is latency-
// bound per k-step — one barrier per k — so it spreads every graph over up to 1024 threads (>= 2 tasks per thread) until the
// launch offers ~48 warps per SM.
static int pick_cluster(int n, int G, bool with_path, int hops, bool want_feat, int *nthreads_out, size_t *smem_out, int *feat_out) {
    for (int C = 1; C <= 8; C *= 2) {
        const int W = k1_W(n, C);
        const int ntask = n * (W / 8);
        // measured (scripts/kbench.py --k1, MOBGT_K1_NT sweeps; n = 128: 2 048 tasks per k-step): 512 threads (4 tasks per thread,
        // two CTAs per SM) beat 256 (8 tasks: 441 / 1 603 us for 256 / 1 024 graphs against 356 / 1 177 us) and 1 024 (one CTA
        // per SM, 410 us); n = 64 is best at 128-256 threads
        int nt = ntask <= 32 ? 32 : ntask <= 128 ? 64 : ntask <= 512 ? 128 : ntask <= 1024 ? 256 : 512;
        // a launch of very few graphs (at most one CTA per SM anyway) is pure k-step latency: spread each graph further
        while (nt < 1024 && 2 * nt <= ntask / 2 + 31 && (long long)G * C <= kNumSMs &&
               k1_smem_bytes(n, C, with_path, 2 * nt, hops, false) <= 227 * 1024)
            nt *= 2;
        if (const char *ev = getenv("MOBGT_K1_NT")) {      // measurement override (scripts/kbench.py)
            const int f = atoi(ev);
            if (f >= 32 && f <= 1024 && (f & (f - 1)) == 0 && f <= ntask * 1 + 31) nt = f;
        }
        const size_t sm = k1_smem_bytes(n, C, with_path, nt, hops, false);
        if (sm <= 227 * 1024) {
            // the feature bytes ride along when they fit and do not halve the CTAs per SM of a small plan
            const size_t smf = k1_smem_bytes(n, C, with_path, nt, hops, true);
            const bool feat = want_feat && smf <= 227 * 1024 && (sm > 100 * 1024 || smf <= 113 * 1024);
            *nthreads_out = nt;
            *smem_out = feat ? smf : sm;
            *feat_out = feat ? 1 : 0;
            return C;
        }
    }
    return -1;
}

// k1_walk_from_path_kernel grid: one thread per pair up to ~4 waves of 256-thread CTAs over the launch (a single graph of a
// per-item call then still spreads over every SM), at least 64 CTAs per graph
static dim3 walk_grid(int n_max, int G) {
    const int cells = n_max * n_max;
    return dim3((unsigned)min(ceil_div(cells, 256), max(64, ceil_div(4 * 8 * kNumSMs, G))), (unsigned)G);
}

// n in (512, MOBGT_MAX_APSP_NODES]: the smallest cluster, 8 (portable) or 16 (non-portable) CTAs, whose M slice fits.
static int pick_cluster_large(int n, size_t *smem_out) {
    for (int C = 8; C <= 16; C *= 2) {
        const size_t sm = k1_large_smem_bytes(n, C);
        if (sm <= 227 * 1024) {
            *smem_out = sm;
            return C;
        }
    }
    return -1;
}

static int32_t apsp_edge_input_large(const K1Params &p, int G_launch, int n_max, cudaStream_t s) {
    MOBGT_REQUIRE(G_launch <= 65535, MOBGT_ERR_BAD_SHAPE, "mobgt_apsp_edge_input: G_launch=%d > 65535 graphs of more than %d nodes",
                  G_launch, MOBGT_MAX_NODES);
    size_t smem = 0;
    const int C = pick_cluster_large(n_max, &smem);
    MOBGT_REQUIRE(C > 0, MOBGT_ERR_UNSUPPORTED, "mobgt_apsp_edge_input: no shared-memory plan for n=%d", n_max);
    auto kern = k1_apsp_large_kernel;
    MOBGT_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    if (C > 8) MOBGT_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3((unsigned)G_launch * C);
    cfg.blockDim = dim3(kLargeThreads);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = s;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = C;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    int resident = 0;
    MOBGT_CUDA_OK(cudaOccupancyMaxActiveClusters(&resident, kern, &cfg));
    MOBGT_REQUIRE(resident >= 1, MOBGT_ERR_UNSUPPORTED,
                  "mobgt_apsp_edge_input: a cluster of %d CTAs x %zu B shared memory (n=%d) cannot be resident on this device",
                  C, smem, n_max);
    MOBGT_CUDA_OK(cudaLaunchKernelEx(&cfg, kern, p, C));
    count_launch();
    if (p.edge_in != nullptr) {
        k1_walk_from_path_kernel<<<walk_grid(n_max, G_launch), 256, 0, s>>>(p.path, p.feat, p.n, p.sq_off, p.gids, p.hops,
                                                                             p.dk, p.shift, p.edge_in);
        MOBGT_LAUNCH_OK("k1_walk_from_path_kernel");
    }
    return MOBGT_OK;
}

}  // namespace mobgt

using namespace mobgt;

extern "C" int32_t mobgt_apsp_edge_input(const uint8_t *feat, const int32_t *n, const int64_t *sq_off,
                                         const int32_t *gids, int32_t G_launch, int32_t n_max_host, int32_t hops,
                                         int32_t dk, int32_t shift, int16_t *dist, int16_t *path, uint8_t *edge_in,
                                         int32_t *maxdist, void *stream) {
    MOBGT_REQUIRE(feat && n && sq_off && dist && maxdist, MOBGT_ERR_NULL, "mobgt_apsp_edge_input: null pointer");
    MOBGT_REQUIRE(G_launch >= 0, MOBGT_ERR_BAD_SHAPE, "mobgt_apsp_edge_input: G_launch=%d", G_launch);
    MOBGT_REQUIRE(n_max_host >= 1 && n_max_host <= MOBGT_MAX_APSP_NODES, MOBGT_ERR_BAD_SHAPE,
                  "mobgt_apsp_edge_input: n_max=%d outside [1,%d]", n_max_host, MOBGT_MAX_APSP_NODES);
    MOBGT_REQUIRE(path != nullptr || n_max_host <= MOBGT_MAX_NODES, MOBGT_ERR_NULL,
                  "mobgt_apsp_edge_input: n_max=%d > %d needs a non-null path buffer (the edge walk reads it)", n_max_host,
                  MOBGT_MAX_NODES);
    MOBGT_REQUIRE(shift == 0 || shift == 1, MOBGT_ERR_BAD_SHAPE, "mobgt_apsp_edge_input: shift must be 0 or 1");
    if (edge_in) {
        MOBGT_REQUIRE(hops >= 4 && hops <= MOBGT_MAX_HOPS && hops % 4 == 0, MOBGT_ERR_UNSUPPORTED,
                      "mobgt_apsp_edge_input: hops=%d must be a multiple of 4 in [4,%d]", hops, MOBGT_MAX_HOPS);
        MOBGT_REQUIRE(dk >= 1 && dk <= hops, MOBGT_ERR_BAD_SHAPE, "mobgt_apsp_edge_input: dk=%d outside [1, hops=%d]", dk, hops);
    } else {
        hops = dk = 4;
    }
    if (G_launch == 0) return MOBGT_OK;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    if (n_max_host > MOBGT_MAX_NODES)
        return apsp_edge_input_large(K1Params{feat, n, sq_off, gids, hops, dk, shift, dist, path, edge_in, maxdist}, G_launch,
                                     n_max_host, s);
    const bool with_path = path != nullptr || n_max_host > MOBGT_UNREACHABLE;   // see skip510 in the kernel
    int nt = 0, feat_in_smem = 0;
    size_t smem = 0;
    const int C = pick_cluster(n_max_host, G_launch, with_path, hops, edge_in != nullptr, &nt, &smem, &feat_in_smem);
    MOBGT_REQUIRE(C > 0, MOBGT_ERR_UNSUPPORTED, "mobgt_apsp_edge_input: no shared-memory plan for n=%d", n_max_host);

    K1Params p{feat, n, sq_off, gids, hops, dk, shift, dist, path, edge_in, maxdist};
    auto kern = with_path ? k1_apsp_kernel<true> : k1_apsp_kernel<false>;
    MOBGT_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3((unsigned)G_launch * C);
    cfg.blockDim = dim3(nt);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = s;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = C;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    MOBGT_CUDA_OK(cudaLaunchKernelEx(&cfg, kern, p, C, feat_in_smem));
    count_launch();
    return MOBGT_OK;
}

extern "C" int32_t mobgt_gen_edge_input(const int16_t *path, const uint8_t *feat, const int32_t *n,
                                        const int64_t *sq_off, int32_t G, int32_t n_max_host, int32_t hops,
                                        int32_t shift, uint8_t *edge_in, void *stream) {
    MOBGT_REQUIRE(path && feat && n && sq_off && edge_in, MOBGT_ERR_NULL, "mobgt_gen_edge_input: null pointer");
    MOBGT_REQUIRE(hops >= 1 && hops <= MOBGT_UNREACHABLE, MOBGT_ERR_BAD_SHAPE, "mobgt_gen_edge_input: hops=%d", hops);
    MOBGT_REQUIRE(n_max_host >= 1 && n_max_host <= MOBGT_MAX_APSP_NODES, MOBGT_ERR_BAD_SHAPE,
                  "mobgt_gen_edge_input: n_max=%d outside [1,%d]", n_max_host, MOBGT_MAX_APSP_NODES);
    if (G <= 0) return MOBGT_OK;
    k1_walk_from_path_kernel<<<walk_grid(n_max_host, G), 256, 0, static_cast<cudaStream_t>(stream)>>>(
        path, feat, n, sq_off, nullptr, hops, hops, shift, edge_in);
    MOBGT_LAUNCH_OK("k1_walk_from_path_kernel");
    return MOBGT_OK;
}

extern "C" int32_t mobgt_degrees(const uint8_t *feat, const int32_t *n, const int64_t *sq_off,
                                 const int64_t *node_off, int32_t G, int32_t shift, int16_t *in_degree,
                                 int16_t *out_degree, void *stream) {
    MOBGT_REQUIRE(feat && n && sq_off && node_off && in_degree && out_degree, MOBGT_ERR_NULL,
                  "mobgt_degrees: null pointer");
    if (G <= 0) return MOBGT_OK;
    k1_degree_kernel<<<G, 128, 0, static_cast<cudaStream_t>(stream)>>>(feat, n, sq_off, node_off, shift, in_degree,
                                                                      out_degree);
    MOBGT_LAUNCH_OK("k1_degree_kernel");
    return MOBGT_OK;
}

// ---- collation helper: pairwise POI distance bin (collator.py:428-437 stand-in for the synthetic world) ----------
// poi_pos[g,i,j] = 1 + min(int(dist(x_i, x_j) / dist_max * (num_bins-2)), num_bins-2), IEEE round-to-nearest single ops in
// the same order as the numpy statement in mobgt_b200/synth.py (PoiWorld.poi_pos_bins), so the bins are bit-identical.
namespace mobgt {
__global__ void k1_poi_pos_kernel(const int32_t *__restrict__ x, const int32_t *__restrict__ n_arr,
                                  const int64_t *__restrict__ sq_off, const int64_t *__restrict__ node_off,
                                  const float *__restrict__ latlon, float dist_max, int num_bins,
                                  int16_t *__restrict__ out) {
    const int g = blockIdx.y;
    const int n = n_arr[g];
    const int64_t so = sq_off[g], no = node_off[g];
    const float scale = (float)(num_bins - 2);
    for (int c = blockIdx.x * blockDim.x + threadIdx.x; c < n * n; c += gridDim.x * blockDim.x) {
        const int i = c / n, j = c - i * n;
        const int a = x[no + i] - 1, b = x[no + j] - 1;
        const float dx = __fsub_rn(latlon[2 * a], latlon[2 * b]);
        const float dy = __fsub_rn(latlon[2 * a + 1], latlon[2 * b + 1]);
        const float d = __fsqrt_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)));
        const float q = __fmul_rn(__fdiv_rn(d, dist_max), scale);
        long long bin = (long long)q;
        if (bin > num_bins - 2) bin = num_bins - 2;
        out[so + c] = (int16_t)(1 + bin);
    }
}
}  // namespace mobgt

extern "C" int32_t mobgt_poi_pos(const int32_t *x, const int32_t *n, const int64_t *sq_off, const int64_t *node_off,
                                 const float *latlon, float dist_max, int32_t num_bins, int32_t G, int32_t n_max_host,
                                 int16_t *poi_pos, void *stream) {
    MOBGT_REQUIRE(x && n && sq_off && node_off && latlon && poi_pos, MOBGT_ERR_NULL, "mobgt_poi_pos: null pointer");
    MOBGT_REQUIRE(num_bins >= 3 && dist_max > 0.f && n_max_host >= 1, MOBGT_ERR_BAD_SHAPE, "mobgt_poi_pos: bad arguments");
    if (G <= 0) return MOBGT_OK;
    dim3 grid((unsigned)min(64, mobgt::ceil_div(n_max_host * n_max_host, 256)), (unsigned)G);
    mobgt::k1_poi_pos_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(x, n, sq_off, node_off, latlon, dist_max,
                                                                                 num_bins, poi_pos);
    MOBGT_LAUNCH_OK("k1_poi_pos_kernel");
    return MOBGT_OK;
}
