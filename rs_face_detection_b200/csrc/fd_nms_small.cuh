// fd_nms_small.cuh — the general single-CTA NMS (K <= 4096: bitonic sort + peel over a 64-bit earlier-overlap mask) as
// device code, shared by nms_cta_kernel / nms_big_kernel's peel (fd_nms.cu) and the fused detect kernel (fd_detect_fused.cu).
#pragma once
#include "fd_internal.cuh"
#include "fd_nms_tiny.cuh"

namespace fd {

constexpr int NT = 1024;          // threads per NMS CTA
constexpr int NWARPS = NT / 32;
constexpr int HEAD = 1024;        // boxes resolved per stage
constexpr int HEAD_WORDS = HEAD / 64;
constexpr int HEAD_MIN = 128;      // initial head of the adaptive peel
constexpr int MASK_WORDS = 64 * (HEAD_WORDS * (HEAD_WORDS + 1) / 2);  // lower-triangular tiles
constexpr int SMALL_CAP = 4096;

// triangular tile layout: tile-row t holds (t+1) 64x64 tiles; inside a tile-row the word index is the slow axis so
// that consecutive rows (lanes) hit consecutive 8-byte words.
__device__ __forceinline__ int mask_index(int i, int w) {
    int t = i >> 6;
    return 64 * (t * (t + 1) / 2) + w * 64 + (i & 63);
}

// ---- head resolve -------------------------------------------------------------------------------------
// Work unit = (tile pair, 16-column quarter, 32-row half): lanes are consecutive rows, the column box is a warp-uniform
// shared-memory broadcast, and each lane writes its own 16-bit piece of the 64-bit mask word (no atomics).
template <int MODE, bool FAST>
__device__ void build_mask(const float4 *__restrict__ hbox, const float *__restrict__ harea, int S, u64 *__restrict__ mask,
                           const IouParams P, int nwarps) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int T = (S + 63) >> 6;
    const int nunits = T * (T + 1) * 4;  // (tile pairs) x 4 quarters x 2 halves
    unsigned short *mask16 = reinterpret_cast<unsigned short *>(mask);
    for (int u = warp; u < nunits; u += nwarps) {
        const int p = u >> 3, q = (u >> 1) & 3, half = u & 1;
        int ti = (int)((sqrtf(8.0f * (float)p + 1.0f) - 1.0f) * 0.5f);
        while ((ti + 1) * (ti + 2) / 2 <= p) ++ti;
        while (ti * (ti + 1) / 2 > p) --ti;
        const int tj = p - ti * (ti + 1) / 2;
        const int i = ti * 64 + half * 32 + lane;
        const int jbase = tj * 64 + q * 16;
        int lane_bound = min(16, S - jbase);                    // columns that exist
        int warp_bound = lane_bound;
        if (ti == tj) {                                         // only earlier boxes j < i
            lane_bound = min(lane_bound, i - jbase);
            warp_bound = min(warp_bound, ti * 64 + half * 32 + 31 - jbase);
        }
        if (i >= S) lane_bound = 0;
        unsigned bits = 0;
        const float4 bi = hbox[min(i, S - 1)];
        const float ai = harea[min(i, S - 1)];
        for (int c = 0; c < warp_bound; ++c) {
            const float4 bj = hbox[jbase + c];
            bool s;
            if (FAST) s = iou_suppresses_exact(bj, harea[jbase + c], bi, ai, P);
            else s = iou_suppresses_full<MODE>(bj, bi, P.thr);
            if (s && c < lane_bound) bits |= (1u << c);
        }
        mask16[(size_t)mask_index(i, tj) * 4 + q] = (unsigned short)bits;
    }
}


// kept/und: HEAD_WORDS words each in shared memory; flags: 2 ints.  On return kept holds the greedy keep set of the head.
// Only the warps that own head rows take part in the rounds (named barrier 1); the rest of the CTA waits at the final
// block-wide barrier, so a round costs a barrier over S threads instead of the whole block.
__device__ inline void resolve_rounds(const u64 *__restrict__ mask, int S, u64 *kept, u64 *und, int *flags) {
    const int i = threadIdx.x;
    if (i < HEAD_WORDS) {
        int lo = i * 64;
        int nbits = min(64, max(0, S - lo));
        und[i] = nbits == 64 ? ~0ull : ((1ull << nbits) - 1ull);
        kept[i] = 0ull;
    }
    if (i == 0) flags[0] = flags[1] = 0;
    __syncthreads();
    const int P = (S + 31) & ~31;  // participating threads (whole warps)
    if (i < P) {
        const int t = i >> 6;
        const u64 bit = 1ull << (i & 63);
        bool undecided = i < S;
        for (int round = 0;; ++round) {
            int dec = 0;  // 0 wait, 1 keep, 2 suppress
            if (undecided) {
                bool sup = false, wait = false;
                for (int w = 0; w <= t; ++w) {
                    u64 e = mask[mask_index(i, w)];
                    if (e & kept[w]) { sup = true; break; }
                    if (e & und[w]) wait = true;
                }
                dec = sup ? 2 : (wait ? 0 : 1);
            }
            named_bar_sync(1, P);  // every read of kept/und of this round (and of last round's flag) is done
            if (i == 0) flags[(round + 1) & 1] = 0;  // next round's flag: last read before the barrier above
            if (dec == 1) atomicOr(&kept[t], bit);
            if (dec != 0) {
                atomicAnd(&und[t], ~bit);
                undecided = false;
            }
            if (undecided) flags[round & 1] = 1;
            named_bar_sync(1, P);
            if (flags[round & 1] == 0) break;
        }
    }
    __syncthreads();
}

// exclusive position of `flag` among the block's threads (thread order) and the block total
__device__ __forceinline__ int block_compact_pos(bool flag, int *warp_sums, int *total, int nwarps) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    unsigned bal = __ballot_sync(0xffffffffu, flag);
    int within = __popc(bal & ((1u << lane) - 1u));
    if (lane == 0) warp_sums[warp] = __popc(bal);
    __syncthreads();
    if (warp == 0) {
        int v = lane < (int)(blockDim.x >> 5) && lane < nwarps ? warp_sums[lane] : 0;
        int incl = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            int n = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += n;
        }
        warp_sums[lane] = incl - v;
        if (lane == 31) warp_sums[32] = incl;
    }
    __syncthreads();
    int pos = warp_sums[warp] + within;
    *total = warp_sums[32];
    __syncthreads();
    return pos;
}

// position of kept bit i inside the kept bitset (ordered) and total count
__device__ __forceinline__ int kept_rank(const u64 *kept, int i, int *total) {
    int pos = 0, tot = 0;
#pragma unroll
    for (int w = 0; w < HEAD_WORDS; ++w) {
        int c = __popcll(kept[w]);
        if (w < (i >> 6)) pos += c;
        tot += c;
    }
    pos += __popcll(kept[i >> 6] & ((1ull << (i & 63)) - 1ull));
    *total = tot;
    return pos;
}

// ---- shared memory carve-up of the single-CTA kernel ------------------------------------------------------
struct SmallSmem {
    float4 sbox[SMALL_CAP];   // boxes in sorted order
    float4 hbox[HEAD];        // current head
    float harea[HEAD];        // areas of the head boxes
    u64 mask[MASK_WORDS];     // also: kept boxes of the head (float4[HEAD] + float[HEAD]) during the push
    u64 keys[SMALL_CAP];      // sort keys; afterwards two int streams [2][SMALL_CAP]
    int sidx[SMALL_CAP];      // source index of sorted rank r
    u64 kept[HEAD_WORDS], und[HEAD_WORDS];
    int warp_sums[33];
    int misc[7];
};

// Box source: `boxes + idx*BS` floats.  BS==4 -> aligned float4 loads.
template <int BS>
__device__ __forceinline__ float4 load_box(const float *__restrict__ boxes, int idx, int stride) {
    if (BS == 4) return __ldg(reinterpret_cast<const float4 *>(boxes) + idx);
    const float *p = boxes + (size_t)idx * stride;
    return make_float4(__ldg(p), __ldg(p + 1), __ldg(p + 2), __ldg(p + 3));
}

struct SmallArgs {
    const u64 *keys;          // [B][key_stride] or nullptr -> keys made from dets scores (column 4)
    size_t key_stride;
    const float *boxes;       // [B][box_batch_stride floats]
    size_t box_batch_stride;
    int box_stride;           // floats between consecutive boxes
    const int *counts;        // [B] or nullptr -> K
    int K;
    int presorted;            // 1 -> input already in pick order (the `_nms` contract): no sort
    int sort_only;            // 1 -> write the sorted source indices and stop (argsort_descending)
    IouParams iou;
    int *keep;                // [B][keep_stride] source indices in pick order
    size_t keep_stride;
    int *keep_count;          // [B]
    int *status;              // [0] NaN flag, [1] number of problems deferred to the big path
    int *big_list;            // problems with K > SMALL_CAP (or nullptr)
    long long *dbg;           // FD_NMS_DBG=1: per-CTA stage timestamps (globaltimer), 16 slots per CTA
    int use_peel;             // FD_NMS_PEEL=1: the peel instead of the mini-head greedy for 1024 < K <= 4096 (A/B reference)
    int no_tiny;              // FD_NMS_NO_TINY=1: force the general single-CTA path for K <= 1024 too (tests, A/B timing)
};


// The general single-CTA path (K <= SMALL_CAP): bitonic sort in shared memory, then the peel.  Called by nms_cta_kernel
// (fd_nms.cu) and, for images with 1024 < K <= 4096 candidates, by the fused detect kernel (fd_detect_fused.cu).  A thread
// that returns early (K <= 256: only 8 warps work; NaN scores) must not meet a later block-wide barrier in the caller.
template <int MODE, int BS>
__device__ void nms_general_cta(const SmallArgs &a, SmallSmem &sm, int b, int K) {
    const int tid = threadIdx.x;
    int *keep = a.keep + (size_t)b * a.keep_stride;
    // Small problems run on 8 warps: whole warps beyond that leave before the first barrier (barriers only count
    // non-exited warps), which makes every block-wide step of the kernel ~4x cheaper for the typical K of a few hundred.
    const int nthr = K <= 256 ? 256 : NT;
    if (tid >= nthr) return;
    const int nwarps = nthr >> 5;
    const float *boxes = a.boxes + (size_t)b * a.box_batch_stride;

    // ---- 1. keys + sort (ascending u64 == score desc, index asc) ----
    int n2 = 2;
    while (n2 < K) n2 <<= 1;
    bool nan_seen = false;
    for (int i = tid; i < n2; i += nthr) {
        u64 key = ~0ull;
        if (i < K) {
            if (a.keys) key = a.keys[(size_t)b * a.key_stride + i];
            else {
                float s = __ldg(boxes + (size_t)i * a.box_stride + 4);
                nan_seen |= (s != s);
                key = ((u64)desc_key(s) << 32) | (unsigned)i;
            }
        }
        sm.keys[i] = key;
    }
    if (__syncthreads_or(nan_seen)) {
        if (tid == 0) {
            atomicExch(&a.status[0], 1);
            a.keep_count[b] = 0;
        }
        return;
    }
    u64 *sorted = sm.keys;
    if (!a.presorted) {
        if (K <= 256) {
            // rank sort (tiny problems only: beyond ~256 keys the bitonic network is cheaper): keys are unique (the index is in the low bits); one key per thread, every thread streams the K
            // keys from shared memory as warp-uniform (broadcast) 128-bit reads and counts the smaller ones
            const u64 mine = tid < K ? sm.keys[tid] : ~0ull;
            int rank = 0;
            const ulonglong2 *k2 = reinterpret_cast<const ulonglong2 *>(sm.keys);
            const int pairs = n2 >> 1;  // padding keys are ~0: never smaller than a real key
            for (int j = 0; j < pairs; ++j) {
                const ulonglong2 q = k2[j];
                rank += (q.x < mine) ? 1 : 0;
                rank += (q.y < mine) ? 1 : 0;
            }
            sorted = sm.keys + SMALL_CAP / 2;
            if (tid < K) sorted[rank] = mine;
            __syncthreads();
        } else {
            for (unsigned k = 2; k <= (unsigned)n2; k <<= 1) {
                for (unsigned j = k >> 1; j > 0; j >>= 1) {
                    for (unsigned t = tid; t < (unsigned)n2 / 2; t += nthr) {
                        unsigned i = ((t & ~(j - 1)) << 1) | (t & (j - 1));
                        unsigned l = i | j;
                        bool up = ((i & k) == 0);
                        u64 x = sm.keys[i], y = sm.keys[l];
                        if ((x > y) == up) {
                            sm.keys[i] = y;
                            sm.keys[l] = x;
                        }
                    }
                    __syncthreads();
                }
            }
        }
    }
    if (a.sort_only) {
        for (int r = tid; r < K; r += nthr) keep[r] = (int)(unsigned)sorted[r];
        if (tid == 0) a.keep_count[b] = K;
        return;
    }

    // ---- 2. gather boxes in sorted order ----
    bool ok = true;
    for (int r = tid; r < K; r += nthr) {
        int idx = (int)(unsigned)sorted[r];
        sm.sidx[r] = idx;
        float4 bx = load_box<BS>(boxes, idx, a.box_stride);
        sm.sbox[r] = bx;
        ok &= box_is_fast_ok(bx);
    }
    const bool fast = __syncthreads_and(ok) && a.iou.fast;  // also fences the key reads before the streams alias them

    if (nthr == NT && !a.use_peel) {
        // ---- 3'. mini-head greedy over up to 4 boxes per thread (fd_nms_tiny.cuh); the peel below stays as the A/B reference ----
        GreedyBufs g;
        float *sarea = reinterpret_cast<float *>(sm.mask);          // the mask region is free on this path
        g.selw = reinterpret_cast<int *>(sarea + SMALL_CAP);
        g.alive = reinterpret_cast<unsigned *>(g.selw + 32 * 32);
        g.mrow = g.alive + 2 * 4 * 32;
        for (int r = tid; r < K; r += nthr) sarea[r] = box_area(sm.sbox[r]);
        __syncthreads();
        g.sbox = sm.sbox;
        g.sarea = sarea;
        g.sidx = sm.sidx;
        int nk;
        if (K <= 2 * NT) nk = fast ? multi_greedy<MODE, true, 2>(g, a.iou, K, keep) : multi_greedy<MODE, false, 2>(g, a.iou, K, keep);
        else nk = fast ? multi_greedy<MODE, true, 4>(g, a.iou, K, keep) : multi_greedy<MODE, false, 4>(g, a.iou, K, keep);
        if (tid == 0) a.keep_count[b] = nk;
        return;
    }
    int *stream_cur = reinterpret_cast<int *>(sm.keys);
    int *stream_nxt = stream_cur + SMALL_CAP;
    float4 *kbox = reinterpret_cast<float4 *>(sm.mask);
    float *karea = reinterpret_cast<float *>(kbox + HEAD);
    bool identity = true;
    int len = K, nk_total = 0;
    // Adaptive head: clustered detections (a few kept boxes suppress everything else) want a small head, because only
    // the KEPT boxes of a head ever touch the rest of the stream; the head doubles while most of it survives.
    const int head_max = min(HEAD, nthr);
    int head_cap = min(HEAD_MIN, head_max);

    // ---- 3. peel ----
    while (len > 0) {
        const int S = min(head_cap, len);
        int my_rank = 0;
        if (tid < S) {
            my_rank = identity ? tid : stream_cur[tid];
            const float4 bx = sm.sbox[my_rank];
            sm.hbox[tid] = bx;
            sm.harea[tid] = box_area(bx);
        }
        __syncthreads();
        if (fast) build_mask<MODE, true>(sm.hbox, sm.harea, S, sm.mask, a.iou, nwarps);
        else build_mask<MODE, false>(sm.hbox, sm.harea, S, sm.mask, a.iou, nwarps);
        __syncthreads();
        resolve_rounds(sm.mask, S, sm.kept, sm.und, sm.misc);
        // (resolve_rounds ends on a block-wide barrier: mask is dead from here, kept is final)
        int nkept = 0;
        bool is_kept = false;
        int pos = 0;
        if (tid < S) {
            is_kept = (sm.kept[tid >> 6] >> (tid & 63)) & 1ull;
            pos = kept_rank(sm.kept, tid, &nkept);
        } else {
            kept_rank(sm.kept, 0, &nkept);
        }
        const int rem = len - S;
        if (is_kept) {
            keep[nk_total + pos] = sm.sidx[my_rank];
            if (rem > 0) {
                kbox[pos] = sm.hbox[tid];
                karea[pos] = sm.harea[tid];
            }
        }
        nk_total += nkept;
        if (2 * nkept > S && head_cap < head_max) head_cap *= 2;
        __syncthreads();
        if (rem <= 0) break;
        int new_len = 0;
        for (int base = 0; base < rem; base += nthr) {
            int r = base + tid;
            bool alive = false;
            int rk = 0;
            if (r < rem) {
                rk = identity ? (S + r) : stream_cur[S + r];
                const float4 bx = sm.sbox[rk];
                alive = true;
                if (fast) {
                    const float ab = box_area(bx);
                    for (int k = 0; k < nkept; ++k)
                        if (iou_suppresses_exact(kbox[k], karea[k], bx, ab, a.iou)) { alive = false; break; }
                } else {
                    for (int k = 0; k < nkept; ++k)
                        if (iou_suppresses_full<MODE>(kbox[k], bx, a.iou.thr)) { alive = false; break; }
                }
            }
            int total;
            int p = block_compact_pos(alive, sm.warp_sums, &total, nwarps);
            if (alive) stream_nxt[new_len + p] = rk;
            new_len += total;
        }
        __syncthreads();
        int *tmp = stream_cur;
        stream_cur = stream_nxt;
        stream_nxt = tmp;
        identity = false;
        len = new_len;
    }
    if (tid == 0) a.keep_count[b] = nk_total;
}

}  // namespace fd
