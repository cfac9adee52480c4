// fd_nms_tiny.cuh — device code of the barrier-light single-CTA NMS for K <= 1024 (shared by nms_cta_kernel in fd_nms.cu
// and the fused post-CNN kernel in fd_detect_fused.cu).  Exact greedy semantics of processing::nms::nms (nms.rs:3-65).
#pragma once
#include "fd_internal.cuh"

namespace fd {

typedef unsigned long long u64;

__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
    asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

// ---- K <= 1024: barrier-light path inside the same kernel --------------------------------------------------------------
// The pipeline's problems are a few hundred candidates of which a few dozen survive; at that size the cost of the general
// path is its ~200 block-wide barriers, not its arithmetic.  Here one thread owns one box:
//   sort     bitonic network on registers: partner distance < 32 by warp shuffle, >= 32 through a double-buffered
//            shared-memory exchange (15 barriers for 1024 keys instead of 55);
//   greedy   the first <= 32 undecided boxes in rank order form a mini-head; its 32 x 32 pairwise tests are one row per warp,
//            every warp then resolves the 32-bit rows redundantly in registers (parallel decision rounds), and every thread
//            tests its own box against the mini-head's kept boxes.  Two barriers per mini-head, no mask in memory, no
//            compaction; nothing is serialised on one warp.
// Same greedy result: a box is kept iff no earlier-ranked kept box suppresses it.
constexpr int TINY_CAP = 1024;
struct TinySmem {
    u64 xch[2][TINY_CAP];
    float4 sbox[TINY_CAP];   // boxes in rank order
    float sarea[TINY_CAP];
    int sidx[TINY_CAP];      // source index of rank r
    int selw[32][32];        // per-warp scratch: ranks of the current mini-head
    unsigned alive[2][32];
    unsigned mrow[32];
    int krank[TINY_CAP];     // rank of the m-th kept box (pick order)
};
__device__ __forceinline__ bool named_bar_or(int id, int nthreads, bool pred) {
    int r;
    asm volatile("{\n\t.reg .pred p, q;\n\tsetp.ne.s32 p, %3, 0;\n\tbar.red.or.pred q, %1, %2, p;\n\tselp.s32 %0, 1, 0, q;\n\t}"
                 : "=r"(r) : "r"(id), "r"(nthreads), "r"((int)pred) : "memory");
    return r != 0;
}
template <int MODE, bool FAST>
__device__ __forceinline__ bool tiny_suppresses(const float4 earlier, const float area_e, const float4 later, const float area_l,
                                                const IouParams &P) {
    if (FAST) return iou_suppresses_exact(earlier, area_e, later, area_l, P);
    return iou_suppresses_full<MODE>(earlier, later, P.thr);
}

template <int MODE, bool FAST>
__device__ int tiny_greedy(TinySmem &sm, const IouParams iou, int K, int nthr, int *keep, float4 my, int *iters_out) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = nthr >> 5;
    const float my_area = box_area(my);
    bool alive = tid < K;
    // the mini-head of the previous round, replicated in every warp: lane j <-> its j-th box
    unsigned keptmask = 0;
    int selj = 0;
    int nk_total = 0, iters = 0;
    for (;; ++iters) {
        // A. my box against the boxes the previous mini-head kept (uniform loop: the shuffles need every lane)
        bool sup = false;
        for (unsigned km = keptmask; km;) {
            const int s0 = __ffs(km) - 1;
            km &= km - 1;
            const int s1 = km ? __ffs(km) - 1 : s0;
            km &= km - 1;   // (0 & anything == 0)
            const int k0 = __shfl_sync(0xffffffffu, selj, s0), k1 = __shfl_sync(0xffffffffu, selj, s1);
            if (alive && !sup) {
                const bool t0 = tiny_suppresses<MODE, FAST>(sm.sbox[k0], sm.sarea[k0], my, my_area, iou);
                const bool t1 = tiny_suppresses<MODE, FAST>(sm.sbox[k1], sm.sarea[k1], my, my_area, iou);
                sup = t0 || t1;
            }
        }
        alive = alive && !sup;
        const unsigned bal = __ballot_sync(0xffffffffu, alive);
        if (lane == 0) sm.alive[iters & 1][warp] = bal;
        named_bar_sync(2, nthr);
        // B. every warp selects the same mini-head: the first <= 32 undecided boxes in rank order
        const unsigned w = lane < nwarps ? sm.alive[iters & 1][lane] : 0u;
        const int c = __popc(w);
        int incl = c;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int n = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += n;
        }
        const int total = __shfl_sync(0xffffffffu, incl, 31);
        if (total == 0) break;
        const int n_sel = min(total, 32);
        int *mysel = sm.selw[warp];
        for (int q = 0, basep = 0; q < nwarps && basep < 32; ++q) {   // all lanes cooperate on one word at a time
            const unsigned wq = __shfl_sync(0xffffffffu, w, q);
            const int p = basep + __popc(wq & ((1u << lane) - 1u));
            if (((wq >> lane) & 1u) && p < 32) mysel[p] = q * 32 + lane;
            basep += __popc(wq);
        }
        __syncwarp();
        selj = lane < n_sel ? mysel[lane] : 0;
        __syncwarp();
        const float4 bj = sm.sbox[selj];
        const float aj = sm.sarea[selj];
        const int warp_excl = __shfl_sync(0xffffffffu, incl - c, warp);   // (not inside the && below: every lane must shuffle)
        const bool selected = alive && (warp_excl + __popc(bal & ((1u << lane) - 1u))) < 32;
        // C. pairwise tests inside the mini-head, one row per warp: bit j of row r = earlier box j suppresses box r
        for (int r = warp; r < n_sel; r += nwarps) {
            const int rs = __shfl_sync(0xffffffffu, selj, r);
            const bool sp = lane < r && tiny_suppresses<MODE, FAST>(bj, aj, sm.sbox[rs], sm.sarea[rs], iou);
            const unsigned row = __ballot_sync(0xffffffffu, sp);
            if (lane == 0) sm.mrow[r] = row;
        }
        named_bar_sync(2, nthr);
        // D. every warp resolves the mini-head by parallel rounds over the 32-bit rows: a box is suppressed as soon as an
        //    earlier overlapping box is kept, kept as soon as every earlier overlapping box is decided (the lowest undecided
        //    box always qualifies, so each round decides at least one; typical dependency depth is 2-3)
        const unsigned m = lane < n_sel ? sm.mrow[lane] : 0u;
        keptmask = __ballot_sync(0xffffffffu, lane < n_sel && m == 0);
        unsigned und = __ballot_sync(0xffffffffu, m != 0);
        bool undecided = m != 0;
        while (und) {
            bool k = false;
            if (undecided) {
                if (m & keptmask) undecided = false;
                else if ((m & und) == 0) { undecided = false; k = true; }
            }
            keptmask |= __ballot_sync(0xffffffffu, k);
            und = __ballot_sync(0xffffffffu, undecided);
        }
        if (warp == 0 && ((keptmask >> lane) & 1u)) {
            const int at = nk_total + __popc(keptmask & ((1u << lane) - 1u));
            keep[at] = sm.sidx[selj];
            sm.krank[at] = selj;
        }
        nk_total += __popc(keptmask);
        if (selected) alive = false;   // decided, one way or the other
    }
    if (iters_out) *iters_out = iters;
    return nk_total;   // identical in every thread
}

// Bitonic network over N2 keys, one per thread, fully unrolled: partner distance < 32 by shuffle, otherwise through the
// double-buffered exchange array (one barrier per such stage).  Used by nms_cta_kernel; the fused detect kernel rank-sorts.
template <int N2>
__device__ __forceinline__ void tiny_sort(u64 &key, TinySmem &sm, int tid) {
    int pbuf = 0;
#pragma unroll
    for (int k = 2; k <= N2; k <<= 1) {
#pragma unroll
        for (int j = k >> 1; j > 0; j >>= 1) {
            u64 other;
            if (j >= 32) {
                sm.xch[pbuf][tid] = key;
                named_bar_sync(2, N2);
                other = sm.xch[pbuf][tid ^ j];
                pbuf ^= 1;
            } else {
                other = __shfl_xor_sync(0xffffffffu, key, j);
            }
            const bool take_min = ((tid & j) == 0) == ((tid & k) == 0);
            key = (take_min == (other < key)) ? other : key;
        }
    }
}


// ---- the same greedy for up to R x 1024 boxes in one CTA of 1024 threads ------------------------------------------------
// Thread t owns the boxes of rank t, t + 1024, ... (so the alive word of its i-th box is word (t >> 5) + 32 i: words are in
// rank order); everything else is tiny_greedy: mini-heads of the first <= 32 undecided boxes, one pairwise row per warp,
// every warp resolving the rows redundantly, every thread testing its R boxes against the mini-head's kept boxes.
// Work ~ K x kept / 1024 tests per thread instead of the peel's mask builds; two block-wide barriers per mini-head.
struct GreedyBufs {
    const float4 *sbox;   // [K] boxes in rank order
    const float *sarea;   // [K]
    const int *sidx;      // [K] source index of rank r
    int *selw;            // [32][32] per-warp scratch
    unsigned *alive;      // [2][R * 32]
    unsigned *mrow;       // [32]
};
template <int MODE, bool FAST, int R>
__device__ int multi_greedy(const GreedyBufs &g, const IouParams iou, int K, int *keep) {
    constexpr int NTH = 1024, NWORDS = R * 32;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    float4 my[R];
    float marea[R];
    bool alive[R];
#pragma unroll
    for (int i = 0; i < R; ++i) {
        const int r = tid + i * NTH;
        alive[i] = r < K;
        my[i] = alive[i] ? g.sbox[r] : make_float4(0.f, 0.f, 0.f, 0.f);
        marea[i] = alive[i] ? g.sarea[r] : 0.f;
    }
    unsigned keptmask = 0;
    int selj = 0, nk_total = 0;
    for (int iters = 0;; ++iters) {
        // A. my boxes against the boxes the previous mini-head kept
        for (unsigned km = keptmask; km; km &= km - 1) {
            const int ks = __shfl_sync(0xffffffffu, selj, __ffs(km) - 1);
            const float4 kb = g.sbox[ks];
            const float ka = g.sarea[ks];
#pragma unroll
            for (int i = 0; i < R; ++i)
                if (alive[i] && tiny_suppresses<MODE, FAST>(kb, ka, my[i], marea[i], iou)) alive[i] = false;
        }
        unsigned *aw = g.alive + (iters & 1) * NWORDS;
#pragma unroll
        for (int i = 0; i < R; ++i) {
            const unsigned bal = __ballot_sync(0xffffffffu, alive[i]);
            if (lane == 0) aw[warp + 32 * i] = bal;
        }
        __syncthreads();
        // B. every warp selects the same mini-head: the first <= 32 undecided boxes in rank order
        int total = 0;
#pragma unroll
        for (int i = 0; i < R; ++i) total += __popc(aw[lane + 32 * i]);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) total += __shfl_xor_sync(0xffffffffu, total, o);
        if (total == 0) break;
        const int n_sel = min(total, 32);
        int *mysel = g.selw + warp * 32;
        for (int q = 0, basep = 0; q < NWORDS && basep < 32; ++q) {
            const unsigned wq = aw[q];
            const int p = basep + __popc(wq & ((1u << lane) - 1u));
            if (((wq >> lane) & 1u) && p < 32) mysel[p] = q * 32 + lane;
            basep += __popc(wq);
        }
        __syncwarp();
        selj = lane < n_sel ? mysel[lane] : 0;
        const int sel_last = mysel[n_sel - 1];   // every undecided box up to this rank is in the mini-head
        __syncwarp();
        const float4 bj = g.sbox[selj];
        const float aj = g.sarea[selj];
        // C. pairwise tests inside the mini-head, one row per warp: bit j of row r = earlier box j suppresses box r
        if (warp < n_sel) {
            const int rs = __shfl_sync(0xffffffffu, selj, warp);
            const bool sp = lane < warp && tiny_suppresses<MODE, FAST>(bj, aj, g.sbox[rs], g.sarea[rs], iou);
            const unsigned row = __ballot_sync(0xffffffffu, sp);
            if (lane == 0) g.mrow[warp] = row;
        }
        __syncthreads();
        // D. every warp resolves the mini-head (parallel decision rounds over the 32-bit rows)
        const unsigned m = lane < n_sel ? g.mrow[lane] : 0u;
        keptmask = __ballot_sync(0xffffffffu, lane < n_sel && m == 0);
        unsigned und = __ballot_sync(0xffffffffu, m != 0);
        bool undecided = m != 0;
        while (und) {
            bool k = false;
            if (undecided) {
                if (m & keptmask) undecided = false;
                else if ((m & und) == 0) { undecided = false; k = true; }
            }
            keptmask |= __ballot_sync(0xffffffffu, k);
            und = __ballot_sync(0xffffffffu, undecided);
        }
        if (warp == 0 && ((keptmask >> lane) & 1u)) keep[nk_total + __popc(keptmask & ((1u << lane) - 1u))] = g.sidx[selj];
        nk_total += __popc(keptmask);
#pragma unroll
        for (int i = 0; i < R; ++i)
            if (tid + i * NTH <= sel_last) alive[i] = false;   // decided, one way or the other
    }
    return nk_total;   // identical in every thread
}

}  // namespace fd
