// fd_nms.cu — stable descending sort + exact greedy IoU NMS, entirely on the device.
//
// Replaces processing::nms::nms (src/processing/nms.rs:3-65), rcnn::cpu_nms (src/rcnn/cpu_nms.rs:10-55) and the
// vestigial CUDA path `_nms` (src/nms_kernel.cu:91-144).  Not a port of the latter: no N x N/64 mask in HBM, no
// D2H mask copy, no CPU sweep.
//
// Algorithm ("peel"): boxes sorted by (score desc, index asc).  The stream of not-yet-removed boxes is consumed
// HEAD (<=1024) boxes at a time.  For a head, a 64-bit "earlier-overlap" mask (row i = bits of earlier head boxes j<i
// with IoU > thr) is built in shared memory; the greedy keep set of the head is then resolved by warp/block-parallel
// rounds over that bitmask (a box is suppressed once an earlier overlapping box is KEPT, kept once all earlier
// overlapping boxes are decided-suppressed) — the same result as the sequential sweep, in O(dependency depth) rounds.
// Only the KEPT boxes of the head are then tested against the rest of the stream, which is compacted in order.
// Work ~ kept x N instead of N^2/2, and nothing larger than the sorted boxes ever touches HBM.
//
//   K <= 1024 : barrier-light single-CTA path (fd_nms_tiny.cuh: register bitonic sort, warp-resolved mini-heads of 32);
//               the batched pipeline runs the same code inside the fused detect kernel (fd_detect_fused.cu).
//   K <= 4096 : one CTA does sort + greedy out of shared memory — per image of a batch (fused detect kernel, nms_batch_*).
//   ONE problem of 1024 < K <= 8192 boxes (fd_nms / fd_nms_device): nms_mid_kernel, a single cooperative launch over all SMs —
//               rank sort, brute-force predecessor lists, the decision sweeps below (72 us at 4 096 boxes, was 178).
//   beyond    : nms_big_kernel, ONE cooperative launch: spatially binned exact NMS without a global sort (boxes binned by cell,
//               ordered inside cells only, predecessor lists + decision sweeps over cell-order positions, kept keys ordered at
//               the end), or — same launch — a radix sort + the cooperative multi-CTA peel for degenerate inputs.  A batch image
//               beyond SMALL_CAP runs the same kernel on the decode kernel's keys (nms_batch_big_image).
//   argsort_descending beyond SMALL_CAP: argsort_kernel, the same launch's radix sort alone.
#include <cooperative_groups.h>
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <cstdio>
#include <vector>
#include "fd_internal.cuh"
#include "fd_nms_tiny.cuh"
#include "fd_nms_small.cuh"

namespace cg = cooperative_groups;

namespace fd {


__device__ __forceinline__ void dbg_stamp(const SmallArgs &a, int slot) {
    if (a.dbg && threadIdx.x == 0 && blockIdx.x < 4096) {   // FD_NMS_DBG=1 keeps the first 4096 problems
        long long t;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
        a.dbg[blockIdx.x * 16 + slot] = t;
    }
}

template <int MODE, int BS>
__device__ void nms_tiny(const SmallArgs &a, unsigned char *smem_raw, int b, int K) {
    TinySmem &sm = *reinterpret_cast<TinySmem *>(smem_raw);
    const int tid = threadIdx.x;
    int n2 = 32;
    while (n2 < K) n2 <<= 1;
    if (tid >= n2) return;   // whole warps; the named barriers below count n2 threads
    const int nthr = n2;
    int *keep = a.keep + (size_t)b * a.keep_stride;
    const float *boxes = a.boxes + (size_t)b * a.box_batch_stride;
    u64 key = ~0ull;
    bool nan_seen = false;
    dbg_stamp(a, 0);
    if (tid < K) {
        if (a.keys) key = a.keys[(size_t)b * a.key_stride + tid];
        else {
            const float s = __ldg(boxes + (size_t)tid * a.box_stride + 4);
            nan_seen = (s != s);
            key = ((u64)desc_key(s) << 32) | (unsigned)tid;
        }
    }
    if (!a.keys && named_bar_or(2, nthr, nan_seen)) {
        if (tid == 0) {
            atomicExch(&a.status[0], 1);
            a.keep_count[b] = 0;
        }
        return;
    }
    if (a.dbg && key == 1) a.dbg[0] = 0;   // (debug) wait for the key load before the stamp
    dbg_stamp(a, 1);
    if (!a.presorted) {
        switch (n2) {
            case 32: tiny_sort<32>(key, sm, tid); break;
            case 64: tiny_sort<64>(key, sm, tid); break;
            case 128: tiny_sort<128>(key, sm, tid); break;
            case 256: tiny_sort<256>(key, sm, tid); break;
            case 512: tiny_sort<512>(key, sm, tid); break;
            default: tiny_sort<1024>(key, sm, tid); break;
        }
    }
    const int idx = (int)(unsigned)key;
    dbg_stamp(a, 2);
    if (a.sort_only) {
        if (tid < K) keep[tid] = idx;
        if (tid == 0) a.keep_count[b] = K;
        return;
    }
    float4 my = make_float4(0.f, 0.f, 0.f, 0.f);
    bool ok = true;
    if (tid < K) {
        my = load_box<BS>(boxes, idx, a.box_stride);
        sm.sbox[tid] = my;
        sm.sarea[tid] = box_area(my);
        sm.sidx[tid] = idx;
        ok = box_is_fast_ok(my);
    }
    const bool fast = !named_bar_or(2, nthr, !ok) && a.iou.fast;   // also publishes sbox / sidx
    dbg_stamp(a, 3);
    int iters = 0;
    const int nk = fast ? tiny_greedy<MODE, true>(sm, a.iou, K, nthr, keep, my, &iters) : tiny_greedy<MODE, false>(sm, a.iou, K, nthr, keep, my, &iters);
    if (tid == 0) a.keep_count[b] = nk;
    dbg_stamp(a, 4);
    if (a.dbg && tid == 0 && blockIdx.x < 4096) { a.dbg[blockIdx.x * 16 + 5] = iters; a.dbg[blockIdx.x * 16 + 6] = K; a.dbg[blockIdx.x * 16 + 7] = nk; }
}

template <int MODE, int BS>
__global__ void __launch_bounds__(NT, 1) nms_cta_kernel(SmallArgs a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    SmallSmem &sm = *reinterpret_cast<SmallSmem *>(smem_raw);
    const int b = blockIdx.x, tid = threadIdx.x;
    const int K = a.counts ? a.counts[b] : a.K;
    int *keep = a.keep + (size_t)b * a.keep_stride;
    if (K <= 0) {
        if (tid == 0) a.keep_count[b] = 0;
        return;
    }
    if (K > SMALL_CAP) {
        if (tid == 0) {
            a.keep_count[b] = -1;
            if (a.big_list) a.big_list[atomicAdd(&a.status[1], 1)] = b;
        }
        return;
    }
    if (K <= TINY_CAP && !a.no_tiny) {
        nms_tiny<MODE, BS>(a, smem_raw, b, K);
        return;
    }
    nms_general_cta<MODE, BS>(a, sm, b, K);
}

// ============================================================================================================
// Big path: cooperative peel (the fallback of nms_big_kernel)
// ============================================================================================================
__global__ void iota_keys_kernel(int n, u64 *__restrict__ keys) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) keys[i] = (u64)(unsigned)i;
}

struct PeelSmem {
    float4 hbox[HEAD];
    float harea[HEAD];
    u64 mask[MASK_WORDS];  // aliased by kbox + karea during push
    u64 kept[HEAD_WORDS], und[HEAD_WORDS];
    int warp_sums[33];
    int red[32];
};

struct PeelArgs {
    const float4 *sbox;
    int N;
    int *stream_a, *stream_b;
    int *keep_ranks;
    int *state;         // [0] scratch, [1] total kept (out), [2] kept of the current stage
    float4 *ks;         // kept boxes of the current stage (HEAD)
    int *tile_counts;   // ceil(N/NT)
    unsigned *ballots;  // ceil(N/NT)*32
    const int *status;  // [2] != 0 -> not fast
    IouParams iou;
};

__device__ __forceinline__ int block_sum(int v, int *red) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if (lane == 0) red[warp] = v;
    __syncthreads();
    int t = red[lane];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
    __syncthreads();
    return t;
}

// The peel itself: every CTA of nms_big_kernel's cooperative grid calls it when the spatial path does not apply.
template <int MODE>
__device__ __forceinline__ void nms_peel_body(const PeelArgs &a, unsigned char *smem_raw) {
    PeelSmem &sm = *reinterpret_cast<PeelSmem *>(smem_raw);
    cg::grid_group grid = cg::this_grid();
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int G = gridDim.x;
    const bool fast = a.iou.fast && (__ldcg(&a.status[2]) == 0);
    float4 *kbox = reinterpret_cast<float4 *>(sm.mask);
    float *karea = reinterpret_cast<float *>(kbox + HEAD);
    int *cur = a.stream_a, *nxt = a.stream_b;
    bool identity = true;
    int len = a.N, nk_total = 0;
    int head_cap = HEAD_MIN;
    while (len > 0) {
        const int S = min(head_cap, len);
        if (blockIdx.x == 0) {
            int my_rank = 0;
            if (tid < S) {
                my_rank = identity ? tid : __ldcg(&cur[tid]);
                const float4 bx = a.sbox[my_rank];
                sm.hbox[tid] = bx;
                sm.harea[tid] = box_area(bx);
            }
            __syncthreads();
            if (fast) build_mask<MODE, true>(sm.hbox, sm.harea, S, sm.mask, a.iou, NWARPS);
            else build_mask<MODE, false>(sm.hbox, sm.harea, S, sm.mask, a.iou, NWARPS);
            __syncthreads();
            resolve_rounds(sm.mask, S, sm.kept, sm.und, sm.red);
            int nkept = 0;
            if (tid < S) {
                bool is_kept = (sm.kept[tid >> 6] >> (tid & 63)) & 1ull;
                int pos = kept_rank(sm.kept, tid, &nkept);
                if (is_kept) {
                    a.keep_ranks[nk_total + pos] = my_rank;
                    a.ks[pos] = sm.hbox[tid];
                }
            } else {
                kept_rank(sm.kept, 0, &nkept);
            }
            if (tid == 0) a.state[2] = nkept;
        }
        grid.sync();
        const int nkept = __ldcg(&a.state[2]);
        nk_total += nkept;
        if (2 * nkept > S && head_cap < HEAD) head_cap *= 2;
        const int rem = len - S;
        if (rem <= 0) break;
        // ---- push: every CTA tests its tiles of the remaining stream against the kept boxes of this stage ----
        for (int k = tid; k < nkept; k += NT) {
            const float4 kb = __ldcg(&a.ks[k]);
            kbox[k] = kb;
            karea[k] = box_area(kb);
        }
        __syncthreads();
        const int ntiles = (rem + NT - 1) / NT;
        for (int t = blockIdx.x; t < ntiles; t += G) {
            int r = t * NT + tid;
            bool alive = false;
            if (r < rem) {
                int rk = identity ? (S + r) : __ldcg(&cur[S + r]);
                float4 bx = a.sbox[rk];
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
            unsigned bal = __ballot_sync(0xffffffffu, alive);
            if (lane == 0) a.ballots[t * 32 + warp] = bal;
            int cnt = __syncthreads_count(alive);
            if (tid == 0) a.tile_counts[t] = cnt;
        }
        grid.sync();
        // ---- ordered scatter of the survivors ----
        int new_len;
        {
            int part = 0;
            for (int t = tid; t < ntiles; t += NT) part += __ldcg(&a.tile_counts[t]);
            new_len = block_sum(part, sm.red);
        }
        for (int t = blockIdx.x; t < ntiles; t += G) {
            int part = 0;
            for (int q = tid; q < t; q += NT) part += __ldcg(&a.tile_counts[q]);
            int offset = block_sum(part, sm.red);
            unsigned myb = __ldcg(&a.ballots[t * 32 + lane]);  // lane w holds the ballot of warp w
            int wpre = 0;
#pragma unroll
            for (int w = 0; w < 32; ++w) {
                unsigned bw = __shfl_sync(0xffffffffu, myb, w);
                if (w < warp) wpre += __popc(bw);
            }
            unsigned mine = __shfl_sync(0xffffffffu, myb, warp);
            if ((mine >> lane) & 1u) {
                int r = t * NT + tid;
                int rk = identity ? (S + r) : __ldcg(&cur[S + r]);
                nxt[offset + wpre + __popc(mine & ((1u << lane) - 1u))] = rk;
            }
        }
        grid.sync();
        int *tmp = cur;
        cur = nxt;
        nxt = tmp;
        identity = false;
        len = new_len;
    }
    if (blockIdx.x == 0 && tid == 0) a.state[1] = nk_total;
}

// ============================================================================================================
// Spatial big path: exact greedy NMS with work proportional to the number of OVERLAPPING pairs.
//
// IoU(A,B) > t implies the intersection is at least t x the larger box in each axis, hence the box centres are at
// most (1-t) x max(w) apart per axis.  Boxes are binned by centre into a uniform grid with that cell size (members of
// a cell ordered by key), every box collects the EARLIER-ranked boxes of its 3x3 neighbourhood that suppress it (exact
// predicate) into a short predecessor list, and the keep set is the unique fixed point of   kept(i) = no predecessor
// kept,   resolved by monotone parallel sweeps inside one cooperative kernel (a box is suppressed as soon as one
// predecessor is kept, kept as soon as all are suppressed).  Same result as the sequential sweep of nms.rs; used when
// every box is regular (finite, positive area), the threshold is an ordinary one and the grid is fine enough —
// otherwise the peel above does the job.
// ============================================================================================================
constexpr int ADJ_CAP = 96;      // mid path: listed predecessors per box (global memory)
constexpr int ADJ_SMEM = 32;     // list entries per box cached in shared memory across sweeps (the big path's lazy lists keep up to 24)
static_assert(ADJ_SMEM >= 24 && ADJ_SMEM % 4 == 0, "the lazy segment loads and the 128-bit list loads rely on this");
constexpr int ADJ_SEG = 64;      // one-launch path: a box's list is three segments of this capacity, one per neighbourhood row (three tasks):
constexpr int ADJ_ROW3 = 3 * ADJ_SEG;   // the first suppressing predecessors of every row.  When all listed ones end up suppressed and there were
                                        // more, the list is refilled (exact; ~40 us each, so the capacity is chosen to make refills rare: at
                                        // 100 000 crowd boxes 16 per row -> 207 boxes overflow and the sweeps take 796 us, 32 -> 5 refills, 77 us,
                                        // 64 -> none, 34 us)
constexpr int GRID_MAX_CELLS = 65535;
constexpr int GRID_MAX_DIM = 4096;

struct GridCfg {
    float minx, miny, cs;
    int gx, gy, use;
};

__device__ __forceinline__ unsigned f2ord(float f) {
    unsigned u = __float_as_uint(f);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float ord2f(unsigned e) {
    unsigned u = (e & 0x80000000u) ? (e & 0x7fffffffu) : ~e;
    return __uint_as_float(u);
}
__device__ __forceinline__ float box_cx(float4 b) { return __fmul_rn(__fadd_rn(b.x, b.z), 0.5f); }
__device__ __forceinline__ float box_cy(float4 b) { return __fmul_rn(__fadd_rn(b.y, b.w), 0.5f); }
__device__ __forceinline__ int cell_coord(float c, float minc, float cs, int g) {
    int v = (int)floorf(__fdiv_rn(__fsub_rn(c, minc), cs));
    return min(g - 1, max(0, v));
}

__device__ __forceinline__ GridCfg grid_setup(unsigned g0, unsigned g1, unsigned g2, unsigned g3, unsigned g4, int N, const IouParams &P, int not_fast) {
    GridCfg c;
    c.minx = ord2f(g0);
    c.miny = ord2f(g1);
    const float maxx = ord2f(g2), maxy = ord2f(g3), maxd = ord2f(g4);
    c.use = 0;
    c.gx = c.gy = 1;
    c.cs = 1.0f;
    if (P.fast && not_fast == 0 && isfinite(maxd) && isfinite(maxx) && isfinite(maxy) && isfinite(c.minx) && isfinite(c.miny)) {
        const float t = fminf(fmaxf(P.thr, 0.0f), 1.0f);
        // centre-distance bound per axis, with a 1% + 0.05 px margin for the separately rounded f32 operations
        double cs = (double)maxd * (1.0 - (double)t) * 1.01 + 0.05;
        const double ex = (double)maxx - (double)c.minx, ey = (double)maxy - (double)c.miny;
        for (int it = 0; it < 64; ++it) {
            double gx = floor(ex / cs) + 1.0, gy = floor(ey / cs) + 1.0;
            if (gx <= GRID_MAX_DIM && gy <= GRID_MAX_DIM && gx * gy <= GRID_MAX_CELLS) {
                c.gx = (int)gx;
                c.gy = (int)gy;
                c.cs = (float)cs;
                // fine enough: on average at most ~2k candidates in a box's 3x3 neighbourhood
                c.use = (9.0 * (double)N / (gx * gy) <= 2048.0) ? 1 : 0;
                break;
            }
            cs *= 1.5;
        }
    }
    return c;
}
// ---- the one-launch path never sorts the boxes globally: boxes are addressed by their position k in
// cell order, members of a cell are ordered by their FULL key (score desc | source index — the order a stable descending sort
// gives), "earlier-ranked" is a key comparison, and the cell of a box is recomputed from its centre.  visit(j) gets a position.
template <class F>
__device__ __forceinline__ void for_each_predecessor_k(int k, const u64 *__restrict__ ckey, const GridCfg &c,
                                                       const int *__restrict__ cell_start, const int *__restrict__ cell_end,
                                                       const float4 *__restrict__ cbox, const float *__restrict__ carea,
                                                       const IouParams &P, F &&visit, int dy0 = -1, int dy1 = 1) {
    const u64 key = ckey[k];
    const float4 bi = cbox[k];
    const float ai = carea[k];
    const int ix = cell_coord(box_cx(bi), c.minx, c.cs, c.gx), iy = cell_coord(box_cy(bi), c.miny, c.cs, c.gy);
    for (int dy = dy0; dy <= dy1; ++dy) {
        const int y = iy + dy;
        if (y < 0 || y >= c.gy) continue;
        for (int dx = -1; dx <= 1; ++dx) {
            const int x = ix + dx;
            if (x < 0 || x >= c.gx) continue;
            const int c2 = y * c.gx + x;
            const int e = cell_end[c2];
            int j = cell_start[c2];
            for (; j + 3 < e; j += 4) {   // members are in key order: 4 candidates per step so their loads are in flight together
                u64 kj[4];
                float4 bj[4];
                float aj[4];
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    kj[u] = ckey[j + u];
                    bj[u] = cbox[j + u];
                    aj[u] = carea[j + u];
                }
                if (kj[0] >= key) break;
#pragma unroll
                for (int u = 0; u < 4; ++u)
                    if (kj[u] < key && iou_suppresses_exact(bj[u], aj[u], bi, ai, P))
                        if (!visit(j + u)) return;
                if (kj[3] >= key) { j = e; break; }
            }
            for (; j < e; ++j) {
                if (ckey[j] >= key) break;
                if (iou_suppresses_exact(cbox[j], carea[j], bi, ai, P))
                    if (!visit(j)) return;
            }
        }
    }
}

__device__ __forceinline__ void adjacency_row_k(int k, int dy, const u64 *__restrict__ ckey, const GridCfg &c, const int *__restrict__ cell_start,
                                                const int *__restrict__ cell_end, const float4 *__restrict__ cbox, const float *__restrict__ carea,
                                                const IouParams &P, int *__restrict__ adj, int *__restrict__ cnt3) {
    int cnt = 0;
    int *mine = adj + (size_t)k * ADJ_ROW3 + (dy + 1) * ADJ_SEG;
    for_each_predecessor_k(k, ckey, c, cell_start, cell_end, cbox, carea, P, [&](int j) {
        if (cnt < ADJ_SEG) mine[cnt] = j;
        ++cnt;
        return cnt <= ADJ_SEG;   // one past the capacity is all the sweeps need to know: stop enumerating
    }, dy, dy);
    cnt3[k * 3 + dy + 1] = cnt;   // ADJ_SEG + 1: more than the segment lists
}

// L2 (cache-global) byte load the compiler may neither cache nor drop: other CTAs update the states concurrently
__device__ __forceinline__ unsigned ld_state(const unsigned char *p) {
    unsigned v;
    asm volatile("ld.global.cg.u8 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}

// Two modes (nms_rounds_body<BRUTE>): the big path's (boxes are cell-order positions, three-segment lists, kept keys appended
// unordered) and the mid path's brute one (boxes are ranks, one list per box from the all-pairs pass, kept source indices
// written in rank order).
struct RoundsArgs {
    int N;
    const u64 *keys;        // keys (score desc | source index) by box: cell order (big path) / rank order (mid path)
    const int *cell_start, *cell_end;   // big path: the grid's cells, cell-ordered boxes and their areas
    const float4 *cbox;
    const float *carea;
    const int *adj, *adj_cnt;
    unsigned char *state;   // by box: 0 undecided, 1 kept, 2 suppressed (zeroed)
    int *counters;          // [3] rotating undecided counters (zeroed)
    int *tile_counts;
    unsigned *ballots;
    int *out_state;         // [1] total kept, [3] grid-wide epochs, [4] list refills (statistics)
    IouParams iou;
    const float4 *sbox;     // brute mode (mid path: no grid): boxes in rank order; a box that exhausts an overflowed list refills it from every earlier box
    int mode;               // brute mode: 0 nms.rs / 1 cpu_nms.rs comparison for the full IEEE test
    const int *status;      // brute mode: [0] NaN score seen, [2] != 0 -> some box is not "fast ok": full IEEE test
    int *final_keep;        // brute mode: kept SOURCE indices in rank order (keys[rank] low word) and {count, NaN flag}
    int *final_num;
    long long *dbg;         // FD_NMS_DBG: globaltimer stamps of block 0 (slots 5..7)
    u64 *kept_keys;         // big path: the kept boxes' keys (unordered) go here; [1] of out_state = count
};

__device__ __forceinline__ void mid_stamp(long long *dbg, int slot) {
    if (dbg && blockIdx.x == 0 && threadIdx.x == 0) {
        long long t;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
        dbg[slot] = t;
    }
}

// FD_NMS_DBG: the latest time any CTA passes a point (slot of the globaltimer stamps)
__device__ __forceinline__ void max_stamp(long long *dbg, int slot) {
    if (dbg && threadIdx.x == 0) {
        long long t;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
        atomicMax(reinterpret_cast<unsigned long long *>(dbg) + slot, (unsigned long long)t);
    }
}

constexpr int ROUND_SWEEPS = 24;   // sweeps of a warp between two grid-wide checks

// brute-mode stand-in for for_each_predecessor_k: every earlier box that suppresses box r
template <class F>
__device__ __forceinline__ void for_each_earlier(int r, const float4 *__restrict__ sbox, const IouParams &P, bool fast, int mode, F &&visit) {
    const float4 bi = __ldcg(sbox + r);
    const float ai = box_area(bi);
    for (int j = 0; j < r; ++j) {
        const float4 bj = __ldcg(sbox + j);
        const bool s = fast ? iou_suppresses_exact(bj, box_area(bj), bi, ai, P)
                            : (mode == 0 ? iou_suppresses_full<0>(bj, bi, P.thr) : iou_suppresses_full<1>(bj, bi, P.thr));
        if (s && !visit(j)) return;
    }
}

// Decides a box from its PENDING predecessors, compacted in place: a suppressed predecessor is final and leaves the list, so
// every sweep polls only what is still undecided (the first visit polls the whole list, later ones a handful).  get(e) / put(e, v)
// access the e-th pending entry.  Returns 0 undecided / 1 kept / 2 suppressed and updates `pend`.
template <class GetFn, class PutFn>
__device__ __forceinline__ int decide_pending(int &pend, GetFn get, PutFn put, const unsigned char *state) {
    int w = 0;
    for (int e = 0; e < pend; e += 8) {
        int id[8];
        unsigned sj[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) id[u] = (e + u < pend) ? get(e + u) : -1;
#pragma unroll
        for (int u = 0; u < 8; ++u) sj[u] = id[u] >= 0 ? ld_state(state + id[u]) : 2u;   // loads in flight together
        bool kept = false;
#pragma unroll
        for (int u = 0; u < 8; ++u) kept |= (sj[u] == 1u);
        if (kept) return 2;
#pragma unroll
        for (int u = 0; u < 8; ++u)
            if (sj[u] == 0u) {   // w <= e + u: never overwrites an entry that has not been read
                put(w, id[u]);
                ++w;
            }
    }
    pend = w;
    return w == 0 ? 1 : 0;
}

// sadj: [ADJ_SMEM][NT] ints of shared memory (head of the pending-predecessor list of each thread's first box, kept across sweeps).
// BRUTE: the mid path's mode (see RoundsArgs).
template <bool BRUTE>
__device__ __forceinline__ void nms_rounds_body(const RoundsArgs &a, const GridCfg &c, int *sadj, int *red) {
    const bool bfast = BRUTE && a.iou.fast && __ldcg(&a.status[2]) == 0;
    cg::grid_group grid = cg::this_grid();
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int G = gridDim.x;
    const int gtid = blockIdx.x * NT + tid, gstride = G * NT;
    volatile unsigned char *state = a.state;
    // ---- prologue: every box's list becomes one compact run of PENDING predecessors (only the listed ones; `overflow` says
    //      there are more) — the resident box of this thread keeps the head of its run in shared memory and the count in a
    //      register, the others (N beyond the resident threads) keep both in global memory: adj_cnt[first counter] = count |
    //      overflow << 30.
    const int cstep = BRUTE ? 1 : 3;
    const int adj_stride = BRUTE ? ADJ_CAP : ADJ_ROW3;   // ints per box in adj
    int *const acnt = const_cast<int *>(a.adj_cnt);
    int *const mine0 = const_cast<int *>(a.adj) + (size_t)min(gtid, max(a.N - 1, 0)) * adj_stride;   // this thread's resident box
    auto get0 = [&](int e) { return e < ADJ_SMEM ? sadj[e * NT + tid] : __ldcg(mine0 + e); };
    auto put0 = [&](int e, int v) {
        if (e < ADJ_SMEM) sadj[e * NT + tid] = v;
        else mine0[e] = v;
    };
    int pend = 0;
    bool overflow = false;
    // Resident box, segmented lists: the segments are consumed LAZILY, up to 8 entries of each at a time (six 128-bit loads in
    // flight together), whenever the pending list runs empty.  Loading every list completely up front cost 15 us at 100 000
    // boxes — as long as the longest list took — although a box with a long list is almost always suppressed by one of its
    // first entries.  At most 24 entries are pending, so the list lives in shared memory and never touches the row again
    // (whose segments still hold what has not been loaded).  segc / segd: listed / loaded entries per segment, 8 bits each.
    unsigned segc = 0, segd = 0;
    auto load_more = [&]() -> bool {
        const int4 *row4 = reinterpret_cast<const int4 *>(mine0);
        int4 q[3][2];
        int rem[3];
#pragma unroll
        for (int sg = 0; sg < 3; ++sg) {
            const int cnt = (segc >> (8 * sg)) & 255, dn = (segd >> (8 * sg)) & 255;
            rem[sg] = min(cnt - dn, 8);
#pragma unroll
            for (int u = 0; u < 2; ++u)
                q[sg][u] = 4 * u < rem[sg] ? __ldcg(row4 + sg * (ADJ_SEG / 4) + (dn >> 2) + u) : make_int4(0, 0, 0, 0);
        }
        bool any = false;
#pragma unroll
        for (int sg = 0; sg < 3; ++sg) {
            const int rm = rem[sg];
            if (rm <= 0) continue;
            any = true;
            const int v[8] = {q[sg][0].x, q[sg][0].y, q[sg][0].z, q[sg][0].w, q[sg][1].x, q[sg][1].y, q[sg][1].z, q[sg][1].w};
#pragma unroll
            for (int i = 0; i < 8; ++i)
                if (i < rm) sadj[(pend++) * NT + tid] = v[i];
            segd += (unsigned)rm << (8 * sg);
        }
        return any;
    };
    const bool lazy = !BRUTE;
    if (lazy && gtid < a.N) {
#pragma unroll
        for (int sg = 0; sg < 3; ++sg) {
            const int cr = __ldcg(&acnt[gtid * 3 + sg]);
            overflow |= cr > ADJ_SEG;
            segc |= (unsigned)min(cr, ADJ_SEG) << (8 * sg);
        }
        load_more();
    }
    for (int r = gtid + (lazy ? gstride : 0); r < a.N; r += gstride) {
        int *row = const_cast<int *>(a.adj) + (size_t)r * adj_stride;
        const int4 *row4 = reinterpret_cast<const int4 *>(row);
        const bool res = r == gtid;
        int total = 0;
        bool ov = false;
        if (!BRUTE) {   // gather the three row segments (typical segment: a few entries, so the three first loads overlap)
            static_assert(ADJ_SEG % 16 == 0, "the gather below loads a segment four 128-bit words at a time");
            int cs[3];
#pragma unroll
            for (int sg = 0; sg < 3; ++sg) {
                const int cr = __ldcg(&acnt[r * 3 + sg]);
                ov |= cr > ADJ_SEG;
                cs[sg] = min(cr, ADJ_SEG);
            }
            int w = 0;
            auto put = [&](int v) { row[w++] = v; };   // w <= the position being read: the gather never overwrites what it has not read
#pragma unroll
            for (int sg = 0; sg < 3; ++sg) {
                for (int g = 0; g * 16 < cs[sg]; ++g) {
                    int4 q[4];
#pragma unroll
                    for (int u = 0; u < 4; ++u)   // in flight together
                        q[u] = 16 * g + 4 * u < cs[sg] ? __ldcg(row4 + sg * (ADJ_SEG / 4) + 4 * g + u) : make_int4(0, 0, 0, 0);
#pragma unroll
                    for (int u = 0; u < 4; ++u) {
                        const int i = 16 * g + 4 * u;
                        if (i < cs[sg]) put(q[u].x);
                        if (i + 1 < cs[sg]) put(q[u].y);
                        if (i + 2 < cs[sg]) put(q[u].z);
                        if (i + 3 < cs[sg]) put(q[u].w);
                    }
                }
            }
            total = w;
        } else {
            const int cr = __ldcg(&acnt[r]);   // (ld.cg throughout: in the mid path the lists were written earlier in this same kernel)
            ov = cr > ADJ_CAP;                  // (mid path: the counter kept running past the list's capacity)
            total = min(cr, ADJ_CAP);
            if (res)
                for (int e = 0; e < min(total, ADJ_SMEM); e += 4) {
                    const int4 q = __ldcg(row4 + (e >> 2));
                    sadj[(e + 0) * NT + tid] = q.x;
                    sadj[(e + 1) * NT + tid] = q.y;
                    sadj[(e + 2) * NT + tid] = q.z;
                    sadj[(e + 3) * NT + tid] = q.w;
                }
        }
        if (res) { pend = total; overflow = ov; }
        else acnt[r * cstep] = total | (ov ? (1 << 30) : 0);
    }
    // A box whose listed predecessors are all suppressed but which has more than the list holds REFILLS its list: it walks its
    // neighbourhood once more, is suppressed if it meets a kept predecessor, and lists the next undecided ones (the suppressed
    // ones, among them everything it has listed before, are final and skipped).  Exact, and rare: by then one of so many
    // predecessors has almost always been kept.  Returns the decision; pn / ov become the new list length and overflow flag.
    auto refill = [&](int r, auto put, int &pn, bool &ov) -> int {
        bool any_kept = false, more = false;
        int w = 0;
        auto visit = [&](int j) {
            const unsigned sj = ld_state(a.state + j);
            if (sj == 1u) { any_kept = true; return false; }
            if (sj == 0u) {
                if (w >= adj_stride) { more = true; return false; }
                put(w, j);
                ++w;
            }
            return true;
        };
        if (BRUTE) for_each_earlier(r, a.sbox, a.iou, bfast, a.mode, visit);
        else for_each_predecessor_k(r, a.keys, c, a.cell_start, a.cell_end, a.cbox, a.carea, a.iou, visit);
        atomicAdd(&a.out_state[4], 1);   // statistics: list refills
        if (any_kept) return 2;
        pn = w;
        ov = more;
        return w == 0 ? 1 : 0;
    };
    __syncthreads();
    max_stamp(a.dbg, 7);    // (slot 11 of the one-launch kernel's timeline: every CTA has loaded its lists)
    bool first_done = gtid >= a.N;
    for (int epoch = 0;; ++epoch) {
        int undecided = 0;
        for (int sweep = 0; sweep < ROUND_SWEEPS; ++sweep) {
            undecided = 0;
            const bool nothing_yet = epoch == 0 && sweep == 0;   // no box is decided yet: polling would read zeros
            if (!first_done) {
                int d = pend == 0 ? 1 : (nothing_yet ? 0 : decide_pending(pend, get0, put0, a.state));
                if (d == 1 && lazy && load_more()) d = 0;   // the listed predecessors seen so far are all suppressed: on to the next ones
                else if (d == 1 && overflow) d = refill(gtid, put0, pend, overflow);
                if (d) {
                    state[gtid] = (unsigned char)d;
                    first_done = true;
                    if (!BRUTE && d == 1) a.kept_keys[atomicAdd(&a.out_state[1], 1)] = __ldcg(&a.keys[gtid]);   // (the caller orders them)
                }
                else ++undecided;
            }
            for (int r = gtid + gstride; r < a.N; r += gstride) {  // only when N exceeds the resident thread count
                if (state[r] != 0) continue;
                const int v = __ldcg(&acnt[r * cstep]);
                int pn = v & 0x3fffffff;
                bool ov = (v >> 30) & 1;
                int *row = const_cast<int *>(a.adj) + (size_t)r * adj_stride;
                auto putr = [&](int e, int x) { row[e] = x; };
                int d = pn == 0 ? 1 : (nothing_yet ? 0 : decide_pending(pn, [&](int e) { return __ldcg(row + e); }, putr, a.state));
                if (d == 1 && ov) d = refill(r, putr, pn, ov);
                if (d == 0 && !nothing_yet) acnt[r * cstep] = pn | (ov ? (1 << 30) : 0);
                if (d) {
                    state[r] = (unsigned char)d;
                    if (!BRUTE && d == 1) a.kept_keys[atomicAdd(&a.out_state[1], 1)] = __ldcg(&a.keys[r]);
                } else ++undecided;
            }
            // Warps sweep at their own pace — no CTA barrier in here, so a warp with short lists advances one dependency link per
            // L2 round trip instead of per (barrier + slowest thread of the CTA).  Measured at 100 000 boxes: CTA-wide sweeps 46 us,
            // the same with two immediate re-polls per sweep 61 us (more polling, same pace), warp-paced sweeps: see DESIGN 4.3.
            if (__all_sync(0xffffffffu, undecided == 0)) break;  // this warp is finished
        }
        int tot = block_sum(undecided, red);
        if (epoch == 0) max_stamp(a.dbg, 8);   // (slot 12: the last CTA leaves the sweeps of the first epoch)
        if (tid == 0 && tot) atomicAdd(&a.counters[epoch % 3], tot);
        __threadfence();
        grid.sync();
        const int left = __ldcg(&a.counters[epoch % 3]);
        if (gtid == 0) {
            a.counters[(epoch + 2) % 3] = 0;
            a.out_state[3] = epoch + 1;  // statistics: grid-wide epochs used
        }
        if (left == 0) break;
    }
    mid_stamp(a.dbg, 5);
    if (!BRUTE) {   // every kept box appended its key when it was decided; the epoch's last grid-wide barrier published them
        mid_stamp(a.dbg, 6);
        return;
    }
    // ordered output of the kept source indices
    const int ntiles = (a.N + NT - 1) / NT;
    for (int t = blockIdx.x; t < ntiles; t += G) {
        const int r = t * NT + tid;
        const bool flag = r < a.N && state[r] == 1;
        unsigned bal = __ballot_sync(0xffffffffu, flag);
        if (lane == 0) a.ballots[t * 32 + warp] = bal;
        int cnt = __syncthreads_count(flag);
        if (tid == 0) a.tile_counts[t] = cnt;
    }
    __threadfence();
    grid.sync();
    for (int t = blockIdx.x; t < ntiles; t += G) {
        int part = 0;
        for (int q = tid; q < t; q += NT) part += __ldcg(&a.tile_counts[q]);
        const int offset = block_sum(part, red);
        const unsigned myb = __ldcg(&a.ballots[t * 32 + lane]);
        int wpre = 0;
#pragma unroll
        for (int w = 0; w < 32; ++w) {
            const unsigned bw = __shfl_sync(0xffffffffu, myb, w);
            if (w < warp) wpre += __popc(bw);
        }
        const unsigned mine = __shfl_sync(0xffffffffu, myb, warp);
        if ((mine >> lane) & 1u) {
            const int pos = offset + wpre + __popc(mine & ((1u << lane) - 1u));
            a.final_keep[pos] = (int)(unsigned)__ldcg(&a.keys[t * NT + tid]);
        }
    }
    if (blockIdx.x == 0) {
        int part = 0;
        for (int q = tid; q < ntiles; q += NT) part += __ldcg(&a.tile_counts[q]);
        const int total = block_sum(part, red);
        if (tid == 0) {
            a.out_state[1] = total;
            a.final_num[0] = total;
            a.final_num[1] = __ldcg(&a.status[0]);
        }
    }
    mid_stamp(a.dbg, 6);
}

// ---- mid path (one problem of a few thousand boxes) ------------------------------------------------------------------
// Between the single-CTA path (one SM's latency chain: 229 us at 4 096 boxes) and the spatial path (nms_big_kernel, built for
// 10^5 boxes) a problem of a few thousand boxes is small enough for brute force over ALL SMs, and short
// enough that launches dominate: separate kernels for these phases measured 103 us at 4 096 boxes, of which ~10 us were
// work.  So the whole problem is ONE cooperative kernel, phases separated by grid-wide barriers, no memset before it:
//   0  clear the status block, ranks, list counters and decision states;
//   1  rank sort: keys (score desc | index) are unique, so rank = number of smaller keys; (row tile x key slice) items count
//      partial ranks, then every box is scattered to its rank (keys and boxes);
//   2  predecessor lists by brute force: (row tile x column tile) items over the lower triangle, N^2/2 exact IoU tests
//      (8.4 M at 4 096 boxes);
//   3  the spatial path's decision sweeps over those lists (nms_rounds_body; a box with more predecessors than a list holds
//      refills it from every earlier box once the listed ones are all suppressed) and its ordered output, written straight as source indices.
constexpr int MID_CAP = 8192;     // measured against nms_big_kernel (host timer): 65.6 vs 83.6 us at 4 096 boxes, 82.0 vs 89.4 at 6 000, 94.3 vs 95.6 at
                                  // 8 192, 166.8 vs 96.0 at 12 288 (against the round-1 launch sequence the crossover was 12 288)
constexpr int MID_CW = 64;        // column tile of phase 2

struct MidArgs {
    const float *dets;
    int n, stride, presorted, mode;
    int slices, per_slice;
    u64 *sorted;
    float4 *sbox;
    int *rank;
    int *st;                // status block (nms_big_kernel's slots), followed by everything that must start at zero
    int zero_ints;
    RoundsArgs ra;
};

__global__ void __launch_bounds__(NT, 1) nms_mid_kernel(MidArgs m) {
    extern __shared__ __align__(16) int dyn[];      // phase 1: key tile; phase 2: column boxes; phase 3: sadj
    __shared__ int red[32];
    cg::grid_group grid = cg::this_grid();
    const int tid = threadIdx.x, G = gridDim.x, gtid = blockIdx.x * NT + tid, gstride = G * NT;
    const int n = m.n;
    mid_stamp(m.ra.dbg, 0);
    for (int i = gtid; i < m.zero_ints; i += gstride) m.st[i] = 0;
    __threadfence();
    grid.sync();
    mid_stamp(m.ra.dbg, 1);
    bool nan_seen = false;
    auto key_of = [&](int j) -> u64 {
        if (m.presorted) return (u64)(unsigned)j;
        const float sc = __ldg(m.dets + (size_t)j * m.stride + 4);
        nan_seen |= (sc != sc);
        return ((u64)desc_key(sc) << 32) | (unsigned)j;
    };
    const int rtiles = (n + NT - 1) / NT;
    if (!m.presorted) {
        u64 *tile = reinterpret_cast<u64 *>(dyn);
        for (int it = blockIdx.x; it < rtiles * m.slices; it += G) {
            const int rt = it / m.slices, sl = it - rt * m.slices;
            const int i = rt * NT + tid;
            const u64 mine = i < n ? key_of(i) : ~0ull;
            const int c0 = sl * m.per_slice, c1 = min(n, c0 + m.per_slice);
            int cnt = 0;
            for (int base = c0; base < c1; base += NT) {
                __syncthreads();
                tile[tid] = base + tid < c1 ? key_of(base + tid) : ~0ull;          // padding: never smaller
                __syncthreads();
                const ulonglong2 *k2 = reinterpret_cast<const ulonglong2 *>(tile);
                const int pairs = (min(NT, c1 - base) + 1) >> 1;
#pragma unroll 4
                for (int j = 0; j < pairs; ++j) {                                  // warp-uniform (broadcast) 128-bit reads
                    const ulonglong2 q = k2[j];
                    cnt += (q.x < mine) ? 1 : 0;
                    cnt += (q.y < mine) ? 1 : 0;
                }
            }
            if (i < n && cnt) atomicAdd(&m.rank[i], cnt);
        }
        __threadfence();
        grid.sync();
    }
    mid_stamp(m.ra.dbg, 2);
    bool ok = true;
    for (int i = gtid; i < n; i += gstride) {
        const u64 key = key_of(i);
        const int r = m.presorted ? i : __ldcg(&m.rank[i]);
        m.sorted[r] = key;
        const float *p = m.dets + (size_t)i * m.stride;
        const float4 bx = make_float4(__ldg(p), __ldg(p + 1), __ldg(p + 2), __ldg(p + 3));
        m.sbox[r] = bx;
        ok &= box_is_fast_ok(bx);
    }
    if (nan_seen) atomicExch(&m.st[0], 1);
    if (!ok) atomicExch(&m.st[2], 1);               // not "fast": the full IEEE overlap test from here on
    __threadfence();
    grid.sync();
    mid_stamp(m.ra.dbg, 3);
    {
        const bool fast = m.ra.iou.fast && __ldcg(&m.st[2]) == 0;
        const IouParams P = m.ra.iou;
        float4 *cb = reinterpret_cast<float4 *>(dyn);
        float *ca = reinterpret_cast<float *>(cb + MID_CW);
        // items = (row tile, column tile) pairs with at least one (row, earlier column): row tile rt has ceil((last row) / CW) of them
        int total_items = 0;
        for (int rt = 0; rt < rtiles; ++rt) total_items += (min(n, (rt + 1) * NT) - 1 + MID_CW - 1) / MID_CW;
        for (int it = blockIdx.x; it < total_items; it += G) {
            int rt = 0, ct = it;
            for (;; ++rt) {
                const int here = (min(n, (rt + 1) * NT) - 1 + MID_CW - 1) / MID_CW;
                if (ct < here) break;
                ct -= here;
            }
            const int j0 = ct * MID_CW, r = rt * NT + tid;
            __syncthreads();
            if (tid < MID_CW && j0 + tid < n) {
                const float4 b = __ldcg(m.sbox + j0 + tid);
                cb[tid] = b;
                ca[tid] = box_area(b);
            }
            __syncthreads();
            if (r >= n) continue;
            const float4 bi = __ldcg(m.sbox + r);
            const float ai = box_area(bi);
            const int lim = min(min(MID_CW, n - j0), r - j0);                      // earlier boxes only
            u64 hits = 0;                                                          // no memory operation inside the test loop
            for (int jj = 0; jj < lim; ++jj) {
                const bool s = fast ? iou_suppresses_exact(cb[jj], ca[jj], bi, ai, P)
                                    : (m.mode == 0 ? iou_suppresses_full<0>(cb[jj], bi, P.thr) : iou_suppresses_full<1>(cb[jj], bi, P.thr));
                hits |= (u64)(s ? 1 : 0) << jj;
            }
            if (hits) {                                                            // items of a row run concurrently: list order is arbitrary
                int pos = atomicAdd(const_cast<int *>(m.ra.adj_cnt) + r, __popcll(hits));
                int *mine = const_cast<int *>(m.ra.adj) + (size_t)r * ADJ_CAP;
                for (; hits && pos < ADJ_CAP; hits &= hits - 1) mine[pos++] = j0 + __ffsll((long long)hits) - 1;
            }
        }
    }
    __threadfence();
    grid.sync();
    mid_stamp(m.ra.dbg, 4);
    nms_rounds_body<true>(m.ra, GridCfg{}, dyn, red);   // (brute mode: no grid)
}

// ---- big path in one launch -------------------------------------------------------------------------------------------
// The spatial path used to be ~25 stream operations (two radix sorts of one kernel per 8-bit pass, nine small kernels, six
// memsets): at 100 000 boxes two thirds of its 332 us were launch gaps and latency-bound 25-CTA radix passes.  nms_big_kernel is
// ONE cooperative kernel, phases separated by grid-wide barriers, and it never sorts the boxes globally:
//   0  keys (score desc | index) made from the scores or taken from the caller, NaN / regularity flags, grid statistics, the
//      OR / NAND of all score keys;
//   1  grid geometry (every CTA, identically); cell of every box and its arrival slot there (atomicAdd);
//   2  cell bounds: scan of the counts;   3  keys to cell order;
//   4  key order inside every cell by counting smaller members; cell-ordered boxes and areas;
//   5  predecessor lists over cell-order positions ("earlier-ranked" = a key comparison);
//   6  decision sweeps (nms_rounds_body) -> the kept boxes' keys, unordered;
//   7  the kept keys ordered by all-pairs counting (radix passes when there are very many) = the reference's output order.
// When the grid does not apply (irregular boxes, degenerate thresholds, too crowded) the same launch sorts globally with the
// cooperative LSD radix sort below (9-bit digits over the index bits of caller keys, then the differing score bits, tiles of
// 1024 keys, per-(digit, tile) counts -> row scans -> stable scatter that also counts the next pass's digits) and runs the peel.
constexpr int CS_BITS = 9;
constexpr int CS_D = 1 << CS_BITS;
constexpr size_t CS_SMEM = sizeof(int) * (size_t)(2 + NWARPS) * CS_D;

struct BigArgs {
    const float *dets;      // box i at dets + i * stride (x1, y1, x2, y2), its score at column 4 when the keys are made here
    int n, stride, presorted, mode;
    const u64 *keys_in;     // optional: the n keys (score desc | box index), in any order (a batch image's, from the decode kernel)
    int ibits;              // bits of the largest box index: the radix passes over the index before the score bits
    u64 *key_e;             // keys by slot e (made: e = the box index); the fallback's sort ping-pongs it with tmp_key
    u64 *tmp_key;           // keys in cell order, arrival order inside a cell
    u64 *ckey;              // keys in cell order, key order inside a cell (final)
    u64 *kept_keys;         // keys of the kept boxes
    int *cell_e, *slot_e;   // cell and arrival slot of the box of key_e[e]
    int *tmp_cell;          // cell of tmp position k
    int *kept_rank;         // rank of a kept key among the kept keys (zero at its first use)
    int *hist;              // fallback / many kept boxes: [2][CS_D][ntiles] digit counts per tile, then [CS_D] digit totals
    float4 *sbox;           // fallback: boxes in rank order
    int *st;                // status block (zero at launch): [0] NaN score, [2] some box not "fast ok", [3] spatial path used, [4] kept,
                            // [5] kept of a peel stage, [6] epochs, [7] list refills, [8..12] grid statistics, [13..15] round counters,
                            // [16..21] GridCfg (statistics), [22] NAND / [23] OR of the score keys, [24] ticket
    int *cell_cnt, *cell_start, *cell_end;
    float4 *cbox;
    float *carea;
    RoundsArgs ra;
    PeelArgs pa;
    int *keep_dev, *keep_count;
    int *nan_flag;          // optional
    long long *dbg;         // FD_NMS_DBG: globaltimer stamps of block 0
};

__device__ __forceinline__ void big_stamp(long long *dbg, int slot) {
    if (dbg && blockIdx.x == 0 && threadIdx.x == 0) {
        long long t;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
        dbg[slot] = t;
    }
}

// digit counts of the tiles this CTA owns, written (not added) to hist[d * ntiles + t]; key(e) yields element e's key
template <class KeyFn>
__device__ __forceinline__ void cs_tile_hist(KeyFn key, int n, int shift, int *__restrict__ hist, int ntiles, int *sh) {
    const int tid = threadIdx.x, lane = tid & 31;
    for (int t = blockIdx.x; t < ntiles; t += gridDim.x) {
        __syncthreads();
        for (int d = tid; d < CS_D; d += NT) sh[d] = 0;
        __syncthreads();
        const int e = t * NT + tid;
        const int d = e < n ? (int)((key(e) >> shift) & (u64)(CS_D - 1)) : CS_D;
        const unsigned peers = __match_any_sync(0xffffffffu, d);
        if (d < CS_D && lane == __ffs(peers) - 1) atomicAdd(&sh[d], __popc(peers));
        __syncthreads();
        for (int dd = tid; dd < CS_D; dd += NT) hist[(size_t)dd * ntiles + t] = sh[dd];
    }
}

// exclusive scan of every digit's counts along the tiles (one warp per digit row), digit totals to tot[]; zeroes `zero` (the
// histogram the scatter that follows accumulates into)
__device__ __forceinline__ void cs_row_scan(int *__restrict__ hist, int *__restrict__ tot, int ntiles, int *__restrict__ zero) {
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int gw = blockIdx.x * NWARPS + warp, nw = gridDim.x * NWARPS;
    for (int d = gw; d < CS_D; d += nw) {
        int *row = hist + (size_t)d * ntiles;
        int carry = 0;
        for (int base = 0; base < ntiles; base += 128) {   // four chunks' loads in flight together
            int v4[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int i = base + u * 32 + lane;
                v4[u] = i < ntiles ? __ldcg(row + i) : 0;
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int i = base + u * 32 + lane;
                int incl = v4[u];
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const int nb = __shfl_up_sync(0xffffffffu, incl, o);
                    if (lane >= o) incl += nb;
                }
                if (i < ntiles) row[i] = carry + incl - v4[u];
                carry += __shfl_sync(0xffffffffu, incl, 31);
            }
        }
        if (lane == 0) tot[d] = carry;
    }
    if (zero) {
        const size_t total = (size_t)CS_D * ntiles;
        for (size_t i = (size_t)blockIdx.x * NT + tid; i < total; i += (size_t)gridDim.x * NT) zero[i] = 0;
    }
}

// stable scatter of one pass: position = digit base + tile base + (warp, lane) order inside the tile
__device__ __forceinline__ void cs_scatter(const u64 *__restrict__ in, u64 *__restrict__ out, int n, int shift, const int *__restrict__ hist_cur,
                                           const int *__restrict__ tot, int *__restrict__ hist_next, int next_shift, int ntiles, int *sh, int *red) {
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    int *dbase = sh, *tbase = sh + CS_D, *wcount = sh + 2 * CS_D;
    __syncthreads();
    {
        const int v = tid < CS_D ? __ldcg(tot + tid) : 0;
        int incl = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int nb = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += nb;
        }
        if (lane == 31) red[warp] = incl;
        __syncthreads();
        int wb = 0;
        for (int w = 0; w < warp; ++w) wb += red[w];
        if (tid < CS_D) dbase[tid] = wb + incl - v;
    }
    for (int t = blockIdx.x; t < ntiles; t += gridDim.x) {
        __syncthreads();
        for (int i = tid; i < NWARPS * CS_D; i += NT) wcount[i] = 0;
        if (tid < CS_D) tbase[tid] = __ldcg(hist_cur + (size_t)tid * ntiles + t);
        __syncthreads();
        const int e = t * NT + tid;
        const bool valid = e < n;
        const u64 key = valid ? __ldcg(in + e) : 0ull;
        const int d = valid ? (int)((key >> shift) & (u64)(CS_D - 1)) : CS_D;
        const unsigned peers = __match_any_sync(0xffffffffu, d);
        const int rank = __popc(peers & ((1u << lane) - 1u));
        if (valid && lane == __ffs(peers) - 1) wcount[warp * CS_D + d] = __popc(peers);
        __syncthreads();
        for (int dd = tid; dd < CS_D; dd += NT) {
            int run = 0;
#pragma unroll 8
            for (int w = 0; w < NWARPS; ++w) {
                const int c = wcount[w * CS_D + dd];
                wcount[w * CS_D + dd] = run;
                run += c;
            }
        }
        __syncthreads();
        int slot = -1;
        if (valid) {
            const int pos = dbase[d] + tbase[d] + wcount[warp * CS_D + d] + rank;
            out[pos] = key;
            if (hist_next) slot = (int)((key >> next_shift) & (u64)(CS_D - 1)) * ntiles + pos / NT;
        }
        if (hist_next) {   // warp-aggregated: neighbouring keys often share the next digit and the destination tile
            const unsigned p2 = __match_any_sync(0xffffffffu, slot);
            if (slot >= 0 && lane == __ffs(p2) - 1) atomicAdd(&hist_next[slot], __popc(p2));
        }
    }
}

// LSD passes over key bits [lo_bit, lo_bit + nbits); hist buffer 0 holds the first pass's counts.  Returns the array that ends
// up sorted (uniform over the grid).  Every CTA must call it.
__device__ __forceinline__ u64 *cs_sort(u64 *a, u64 *b, int n, int lo_bit, int nbits, int *hist, int ntiles, int *sh, int *red) {
    cg::grid_group grid = cg::this_grid();
    const size_t hsz = (size_t)CS_D * ntiles;
    int *tot = hist + 2 * hsz;
    const int npass = (nbits + CS_BITS - 1) / CS_BITS;
    u64 *in = a, *out = b;
    for (int p = 0; p < npass; ++p) {
        int *hcur = hist + (size_t)(p & 1) * hsz, *hnext = hist + (size_t)((p + 1) & 1) * hsz;
        const bool more = p + 1 < npass;
        cs_row_scan(hcur, tot, ntiles, more ? hnext : nullptr);
        __threadfence();
        grid.sync();
        cs_scatter(in, out, n, lo_bit + CS_BITS * p, hcur, tot, more ? hnext : nullptr, lo_bit + CS_BITS * (p + 1), ntiles, sh, red);
        __threadfence();
        grid.sync();
        u64 *tmp = in;
        in = out;
        out = tmp;
    }
    return in;
}

// Sorts n unique keys: LSD passes over the index bits [0, ibits) — 0 when the keys are already in index order — then over the
// score bits that differ (diff: a mask of the high-word bits in which the keys differ).  Returns the sorted array; every CTA must call it.
__device__ __forceinline__ u64 *cs_sort_keys(u64 *a, u64 *b, int n, int ibits, unsigned diff, int *hist, int *sh, int *red) {
    cg::grid_group grid = cg::this_grid();
    const int ntiles = (n + NT - 1) / NT;
    if (ibits > 0) {
        cs_tile_hist([&](int e) { return __ldcg(a + e); }, n, 0, hist, ntiles, sh);
        __threadfence();
        grid.sync();
        u64 *r = cs_sort(a, b, n, 0, ibits, hist, ntiles, sh, red);
        if (r != a) { b = a; a = r; }
    }
    const int nbits = diff ? 32 - __clz(diff) : 0;
    if (nbits > 0) {
        cs_tile_hist([&](int e) { return __ldcg(a + e); }, n, 32, hist, ntiles, sh);
        __threadfence();
        grid.sync();
        a = cs_sort(a, b, n, 32, nbits, hist, ntiles, sh, red);
    }
    return a;
}

__device__ __forceinline__ unsigned differing_score_bits(const int *nand_or) {   // from the NAND and the OR of all score keys
    return (~__ldcg(reinterpret_cast<const unsigned *>(nand_or))) ^ __ldcg(reinterpret_cast<const unsigned *>(nand_or) + 1);
}

constexpr int KEPT_RANK_CAP = 16384;   // kept keys ordered by all-pairs counting up to here (6 357 at 100 000 boxes), by the radix passes beyond

__global__ void __launch_bounds__(NT, 1) nms_big_kernel(BigArgs m) {
    extern __shared__ __align__(16) int dyn[];
    __shared__ int red[32];
    __shared__ GridCfg scfg;
    cg::grid_group grid = cg::this_grid();
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, G = gridDim.x, gtid = blockIdx.x * NT + tid, gstride = G * NT;
    const int n = m.n;
    unsigned *gs = reinterpret_cast<unsigned *>(m.st + 8);
    big_stamp(m.dbg, 0);
    // ---- 0. keys, flags, grid statistics; arrays that must start at zero ----
    {
        unsigned acc_or = 0, acc_nand = 0;
        unsigned mincx = 0xFFFFFFFFu, mincy = 0xFFFFFFFFu, maxcx = 0, maxcy = 0, maxd = 0;
        bool nan_seen = false, ok = true;
        for (int e = gtid; e < n; e += gstride) {
            u64 key;
            if (m.keys_in) {
                key = __ldg(m.keys_in + e);   // (no NaN check: the decode kernel drops NaN scores)
            } else if (m.presorted) {
                key = (u64)(unsigned)e;
            } else {
                const float sc = __ldg(m.dets + (size_t)e * m.stride + 4);
                nan_seen |= (sc != sc);
                key = ((u64)desc_key(sc) << 32) | (unsigned)e;
            }
            m.key_e[e] = key;
            const unsigned k32 = (unsigned)(key >> 32);
            acc_or |= k32;
            acc_nand |= ~k32;
            const float *p = m.dets + (size_t)(unsigned)key * m.stride;
            const float4 b = make_float4(__ldg(p), __ldg(p + 1), __ldg(p + 2), __ldg(p + 3));
            ok &= box_is_fast_ok(b);
            const unsigned cx = f2ord(box_cx(b)), cy = f2ord(box_cy(b));
            mincx = min(mincx, cx); maxcx = max(maxcx, cx);
            mincy = min(mincy, cy); maxcy = max(maxcy, cy);
            const float w = __fadd_rn(__fsub_rn(b.z, b.x), 1.0f), h = __fadd_rn(__fsub_rn(b.w, b.y), 1.0f);
            maxd = max(maxd, f2ord(fmaxf(fabsf(w), fabsf(h))));
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            acc_or |= __shfl_xor_sync(0xffffffffu, acc_or, o);
            acc_nand |= __shfl_xor_sync(0xffffffffu, acc_nand, o);
            mincx = min(mincx, __shfl_xor_sync(0xffffffffu, mincx, o));
            mincy = min(mincy, __shfl_xor_sync(0xffffffffu, mincy, o));
            maxcx = max(maxcx, __shfl_xor_sync(0xffffffffu, maxcx, o));
            maxcy = max(maxcy, __shfl_xor_sync(0xffffffffu, maxcy, o));
            maxd = max(maxd, __shfl_xor_sync(0xffffffffu, maxd, o));
        }
        unsigned *ured = reinterpret_cast<unsigned *>(dyn);   // one set of atomics per CTA, not per warp
        if (lane == 0) {
            ured[warp] = acc_or; ured[32 + warp] = acc_nand;
            ured[64 + warp] = mincx; ured[96 + warp] = mincy; ured[128 + warp] = maxcx; ured[160 + warp] = maxcy; ured[192 + warp] = maxd;
        }
        __syncthreads();
        if (tid < 32) {
            acc_or = ured[tid]; acc_nand = ured[32 + tid];
            mincx = ured[64 + tid]; mincy = ured[96 + tid]; maxcx = ured[128 + tid]; maxcy = ured[160 + tid]; maxd = ured[192 + tid];
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                acc_or |= __shfl_xor_sync(0xffffffffu, acc_or, o);
                acc_nand |= __shfl_xor_sync(0xffffffffu, acc_nand, o);
                mincx = min(mincx, __shfl_xor_sync(0xffffffffu, mincx, o));
                mincy = min(mincy, __shfl_xor_sync(0xffffffffu, mincy, o));
                maxcx = max(maxcx, __shfl_xor_sync(0xffffffffu, maxcx, o));
                maxcy = max(maxcy, __shfl_xor_sync(0xffffffffu, maxcy, o));
                maxd = max(maxd, __shfl_xor_sync(0xffffffffu, maxd, o));
            }
            if (tid == 0) {
                if (acc_or | acc_nand) {
                    atomicOr(reinterpret_cast<unsigned *>(m.st) + 22, acc_nand);
                    atomicOr(reinterpret_cast<unsigned *>(m.st) + 23, acc_or);
                }
                if (mincx != 0xFFFFFFFFu) {   // (a CTA without boxes has nothing to report)
                    // min cx / min cy are kept complemented so that the memset's zero is their identity as well
                    atomicMax(&gs[0], ~mincx);
                    atomicMax(&gs[1], ~mincy);
                    atomicMax(&gs[2], maxcx);
                    atomicMax(&gs[3], maxcy);
                    atomicMax(&gs[4], maxd);
                }
            }
        }
        if (__syncthreads_or(nan_seen) && tid == 0) atomicExch(&m.st[0], 1);
        if (__syncthreads_or(!ok) && tid == 0) atomicExch(&m.st[2], 1);
        unsigned *state4 = reinterpret_cast<unsigned *>(m.ra.state);
        for (int i = gtid; i < (n + 3) / 4; i += gstride) state4[i] = 0u;
        for (int i = gtid; i <= GRID_MAX_CELLS; i += gstride) m.cell_cnt[i] = 0;
        for (int i = gtid; i < n; i += gstride) m.kept_rank[i] = 0;
    }
    __threadfence();
    grid.sync();
    big_stamp(m.dbg, 1);
    // ---- grid geometry: every CTA derives the same one ----
    if (tid == 0) {
        scfg = grid_setup(~__ldcg(gs + 0), ~__ldcg(gs + 1), __ldcg(gs + 2), __ldcg(gs + 3), __ldcg(gs + 4), n, m.ra.iou, __ldcg(&m.st[2]));
        if (blockIdx.x == 0) {
            *reinterpret_cast<GridCfg *>(m.st + 16) = scfg;
            m.st[3] = scfg.use;
        }
    }
    __syncthreads();
    const GridCfg c = scfg;
    if (!c.use) {
        // ---- the grid does not apply (irregular boxes, degenerate threshold, too crowded; uniform over the launch): global sort by
        //      key (made keys are in index order already, so their sort passes over the score bits only), boxes in rank order,
        //      the peel, and its kept ranks become source indices ----
        u64 *sorted = cs_sort_keys(m.key_e, m.tmp_key, n, m.keys_in ? m.ibits : 0, differing_score_bits(m.st + 22), m.hist, dyn, red);
        for (int r = gtid; r < n; r += gstride) {
            const int idx = (int)(unsigned)__ldcg(sorted + r);
            const float *p = m.dets + (size_t)idx * m.stride;
            m.sbox[r] = make_float4(__ldg(p), __ldg(p + 1), __ldg(p + 2), __ldg(p + 3));
        }
        __threadfence();
        grid.sync();
        if (m.mode == 0) nms_peel_body<0>(m.pa, reinterpret_cast<unsigned char *>(dyn));
        else nms_peel_body<1>(m.pa, reinterpret_cast<unsigned char *>(dyn));
        __threadfence();
        grid.sync();
        const int total = __ldcg(&m.pa.state[1]);
        for (int k = gtid; k < total; k += gstride) m.keep_dev[k] = (int)(unsigned)__ldcg(sorted + __ldcg(&m.pa.keep_ranks[k]));
        if (gtid == 0) {
            *m.keep_count = total;
            if (m.nan_flag) *m.nan_flag = __ldcg(&m.st[0]);
        }
        return;
    }
    const int ncells = c.gx * c.gy;
    // ---- 1. cell of every box and its arrival slot there (no global sort: only the members of a cell get ordered) ----
    for (int e = gtid; e < n; e += gstride) {
        const float *p = m.dets + (size_t)(unsigned)m.key_e[e] * m.stride;   // (key_e[e] was written by this very thread in phase 0)
        const float4 b = make_float4(__ldg(p), __ldg(p + 1), __ldg(p + 2), __ldg(p + 3));
        const int cell = cell_coord(box_cy(b), c.miny, c.cs, c.gy) * c.gx + cell_coord(box_cx(b), c.minx, c.cs, c.gx);
        m.cell_e[e] = cell;
        m.slot_e[e] = atomicAdd(&m.cell_cnt[cell], 1);
    }
    __threadfence();
    grid.sync();
    big_stamp(m.dbg, 2);
    // ---- 2. cell bounds: exclusive scan of the counts; every CTA sums what precedes its chunk of cells and scans the chunk ----
    {
        const int per = (ncells + G - 1) / G;   // <= 443 cells per CTA
        const int c0 = min(ncells, (int)blockIdx.x * per), c1 = min(ncells, c0 + per);
        int part = 0;
        for (int i = tid; i < c0; i += NT) part += __ldcg(&m.cell_cnt[i]);
        int before = block_sum(part, red);
        for (int base = c0; base < c1; base += NT) {   // (one round on a 148-SM part: at most 443 cells per CTA)
            const int i = base + tid;
            const int v = i < c1 ? __ldcg(&m.cell_cnt[i]) : 0;
            int incl = v;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int nb = __shfl_up_sync(0xffffffffu, incl, o);
                if (lane >= o) incl += nb;
            }
            __syncthreads();
            if (lane == 31) red[warp] = incl;
            __syncthreads();
            int wb = 0;
            for (int w = 0; w < warp; ++w) wb += red[w];
            if (i < c1) {
                const int start = before + wb + incl - v;
                m.cell_start[i] = start;
                m.cell_end[i] = start + v;
            }
            for (int w = 0; w < NWARPS; ++w) before += red[w];
        }
    }
    __threadfence();
    grid.sync();
    big_stamp(m.dbg, 3);
    // ---- 3. keys to cell order (arrival order inside a cell) ----
    for (int e = gtid; e < n; e += gstride) {
        const int cell = m.cell_e[e];                       // (written by this very thread in phase 1)
        const int k = __ldcg(&m.cell_start[cell]) + m.slot_e[e];
        m.tmp_key[k] = m.key_e[e];
        m.tmp_cell[k] = cell;
    }
    __threadfence();
    grid.sync();
    big_stamp(m.dbg, 4);
    // ---- 4. key order inside every cell (position = number of smaller keys among the cell's members), cell-ordered boxes ----
    for (int k = gtid; k < n; k += gstride) {
        const int cell = __ldcg(&m.tmp_cell[k]);
        const int cs = __ldcg(&m.cell_start[cell]), ce = __ldcg(&m.cell_end[cell]);
        // (L1-cached loads: the threads of a cell read the same members, and no SM has read tmp_key through L1 before this phase)
        const u64 mine = m.tmp_key[k];
        int cnt = 0, j = cs;
        for (; j + 3 < ce; j += 4) {
            const u64 k0 = m.tmp_key[j], k1 = m.tmp_key[j + 1], k2 = m.tmp_key[j + 2], k3 = m.tmp_key[j + 3];
            cnt += (k0 < mine) + (k1 < mine) + (k2 < mine) + (k3 < mine);
        }
        for (; j < ce; ++j) cnt += m.tmp_key[j] < mine;
        const int pos = cs + cnt;
        const float *p = m.dets + (size_t)(unsigned)mine * m.stride;
        const float4 b = make_float4(__ldg(p), __ldg(p + 1), __ldg(p + 2), __ldg(p + 3));
        m.ckey[pos] = mine;
        m.cbox[pos] = b;
        m.carea[pos] = box_area(b);
    }
    __threadfence();
    grid.sync();
    big_stamp(m.dbg, 5);
    // ---- 5. predecessor lists ----
    {   // (box, neighbourhood row) tasks, row-major so a warp's lanes are consecutive cell-ordered boxes on the same row; warps take
        // 32 tasks at a time from a ticket (rows and cells differ in cost).  Measured at 100 000 boxes: one box per thread in
        // contiguous chunks 145 us, 256-box tiles dealt round-robin 124, whole boxes from a ticket 119, these row tasks 82;
        // one warp per (non-empty cell, row) — lanes walking the same candidate cells — 151 (few, uneven tasks).
        int *ticket = m.st + 24;
        const long long tasks = 3ll * n;
        for (;;) {
            int base = 0;
            if (lane == 0) base = atomicAdd(ticket, 32);
            base = __shfl_sync(0xffffffffu, base, 0);
            if (base >= tasks) break;
            const int q = base + lane;
            if (q < tasks) {
                const int row = q / n, k = q - row * n;
                adjacency_row_k(k, row - 1, m.ckey, c, m.cell_start, m.cell_end, m.cbox, m.carea, m.ra.iou, const_cast<int *>(m.ra.adj), const_cast<int *>(m.ra.adj_cnt));
            }
        }
    }
    __threadfence();
    grid.sync();
    big_stamp(m.dbg, 6);
    // ---- 6. decision sweeps; the kept boxes' keys come out in position order ----
    RoundsArgs ra = m.ra;
    ra.dbg = m.dbg ? m.dbg + 4 : nullptr;   // its stamps 5 / 6 land in slots 9 / 10
    nms_rounds_body<false>(ra, c, dyn, red);   // (ends behind the grid-wide barrier of its last epoch: kept keys and their count are visible)
    big_stamp(m.dbg, 7);
    // ---- 7. the kept keys in key order = the reference's output order ----
    const int M = __ldcg(&m.st[4]);
    if (M <= KEPT_RANK_CAP) {   // rank = number of smaller kept keys: (row tile x key slice) items count partial ranks
        const int rtiles = (M + NT - 1) / NT;
        int slices = max(1, min(G / max(rtiles, 1), (M + 127) / 128));   // one item per CTA where possible
        const int per_slice = (((M + slices - 1) / slices) + 1) & ~1;
        slices = per_slice > 0 ? (M + per_slice - 1) / per_slice : 0;
        u64 *tile = reinterpret_cast<u64 *>(dyn);
        for (int it = blockIdx.x; it < rtiles * slices; it += G) {
            const int rt = it / slices, sl = it - rt * slices;
            const int i = rt * NT + tid;
            const u64 mine = i < M ? __ldcg(&m.kept_keys[i]) : ~0ull;
            const int s0 = sl * per_slice, s1 = min(M, s0 + per_slice);
            int cnt = 0;
            for (int base = s0; base < s1; base += NT) {
                __syncthreads();
                tile[tid] = base + tid < s1 ? __ldcg(&m.kept_keys[base + tid]) : ~0ull;   // padding: never smaller
                __syncthreads();
                const ulonglong2 *k2 = reinterpret_cast<const ulonglong2 *>(tile);
                const int pairs = (min(NT, s1 - base) + 1) >> 1;
#pragma unroll 4
                for (int j = 0; j < pairs; ++j) {   // warp-uniform (broadcast) 128-bit reads
                    const ulonglong2 q = k2[j];
                    cnt += (q.x < mine) ? 1 : 0;
                    cnt += (q.y < mine) ? 1 : 0;
                }
            }
            if (i < M && cnt) atomicAdd(&m.kept_rank[i], cnt);
        }
        __threadfence();
        grid.sync();
        for (int i = gtid; i < M; i += gstride) m.keep_dev[__ldcg(&m.kept_rank[i])] = (int)(unsigned)__ldcg(&m.kept_keys[i]);
    } else {                    // very many kept boxes (appended in no particular order): radix passes over index and score bits
        const u64 *sorted = cs_sort_keys(m.kept_keys, m.tmp_key, M, m.ibits, differing_score_bits(m.st + 22), m.hist, dyn, red);
        for (int i = gtid; i < M; i += gstride) m.keep_dev[i] = (int)(unsigned)__ldcg(sorted + i);
    }
    if (gtid == 0) {
        *m.keep_count = M;
        if (m.nan_flag) *m.nan_flag = __ldcg(&m.st[0]);
    }
    big_stamp(m.dbg, 8);
}

// argsort_descending beyond SMALL_CAP: keys (score desc | index) from the score column alone — the caller passes (scores - 4)
// with stride 1, so any other column would be another score or the pad — sorted by nms_big_kernel's radix passes over the
// differing score bits (the keys are made in index order, so ties stay stable).  st (zero at launch): [0] NaN score seen,
// [1] NAND / [2] OR of the score keys.
__global__ void __launch_bounds__(NT, 1) argsort_kernel(const float *__restrict__ dets, int n, int stride, u64 *keys, u64 *tmp, int *hist,
                                                        int *st, int *__restrict__ order, int *__restrict__ flag) {
    extern __shared__ __align__(16) int dyn[];
    __shared__ int red[32];
    __shared__ unsigned acc[2];
    cg::grid_group grid = cg::this_grid();
    const int tid = threadIdx.x, gtid = blockIdx.x * NT + tid, gstride = gridDim.x * NT;
    if (tid == 0) acc[0] = acc[1] = 0u;
    __syncthreads();
    unsigned acc_or = 0, acc_nand = 0;
    bool nan_seen = false;
    for (int e = gtid; e < n; e += gstride) {
        const float sc = __ldg(dets + (size_t)e * stride + 4);
        nan_seen |= (sc != sc);
        const unsigned k32 = desc_key(sc);
        keys[e] = ((u64)k32 << 32) | (unsigned)e;
        acc_or |= k32;
        acc_nand |= ~k32;
    }
    acc_or = __reduce_or_sync(0xffffffffu, acc_or);
    acc_nand = __reduce_or_sync(0xffffffffu, acc_nand);
    if ((tid & 31) == 0) {   // one pair of global atomics per CTA
        atomicOr(&acc[0], acc_nand);
        atomicOr(&acc[1], acc_or);
    }
    if (__syncthreads_or(nan_seen) && tid == 0) atomicExch(&st[0], 1);
    if (tid == 0 && (acc[0] | acc[1])) {
        atomicOr(reinterpret_cast<unsigned *>(st) + 1, acc[0]);
        atomicOr(reinterpret_cast<unsigned *>(st) + 2, acc[1]);
    }
    __threadfence();
    grid.sync();
    const u64 *sorted = cs_sort_keys(keys, tmp, n, 0, differing_score_bits(st + 1), hist, dyn, red);
    for (int r = gtid; r < n; r += gstride) order[r] = (int)(unsigned)__ldcg(sorted + r);
    if (gtid == 0) *flag = __ldcg(&st[0]);
}

// ---- host side ------------------------------------------------------------------------------------------------
// Decision boundary of the exact division-free test (see iou_suppresses_exact).
IouParams make_iou_params(float thr, int mode) {
    IouParams p;
    p.thr = thr;
    p.m = 0.0;
    p.incl = 0;
    p.fast = 0;
    if (!(thr == thr) || std::isinf(thr) || thr > 1e30f) return p;
    uint32_t bits;
    memcpy(&bits, &thr, 4);
    if (mode == 0) {          // suppress iff fl(q) > thr  <=>  fl(q) >= next(thr)
        if (thr < 0.0f) return p;
        float nxt = nextafterf(thr, INFINITY);
        uint32_t nb;
        memcpy(&nb, &nxt, 4);
        p.m = ((double)thr + (double)nxt) * 0.5;
        p.incl = (nb & 1u) == 0;   // a tie rounds to the even neighbour: next(thr) when it is even
        p.fast = 1;
    } else {                  // suppress iff fl(q) >= thr
        if (!(thr > 0.0f)) return p;
        float prv = nextafterf(thr, -INFINITY);
        p.m = ((double)prv + (double)thr) * 0.5;
        p.incl = (bits & 1u) == 0; // tie rounds to thr when thr is even
        p.fast = 1;
    }
    return p;
}

template <int MODE>
static int launch_small(fd_ctx *ctx, const SmallArgs &a_in, int B, bool float4_boxes) {
    static const int no_tiny = getenv("FD_NMS_NO_TINY") != nullptr && getenv("FD_NMS_NO_TINY")[0] == '1';
    SmallArgs a = a_in;
    a.no_tiny = no_tiny;
    static const int use_peel = getenv("FD_NMS_PEEL") != nullptr && getenv("FD_NMS_PEEL")[0] == '1';
    a.use_peel = use_peel;
    static const int dbg_on = getenv("FD_NMS_DBG") != nullptr;
    static long long *dbg_dev = nullptr;
    if (dbg_on) {
        if (!dbg_dev) FD_CUDA(cudaMalloc(&dbg_dev, sizeof(long long) * 16 * 4096));
        FD_CUDA(cudaMemsetAsync(dbg_dev, 0, sizeof(long long) * 16 * 4096, ctx->stream));
        a.dbg = dbg_dev;
    }
    static_assert(sizeof(TinySmem) <= sizeof(SmallSmem), "tiny path lives in the general path's shared memory");
    const size_t smem = sizeof(SmallSmem);
    if (float4_boxes) {
        FD_CUDA(cudaFuncSetAttribute(nms_cta_kernel<MODE, 4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        nms_cta_kernel<MODE, 4><<<B, NT, smem, ctx->stream>>>(a);
    } else {
        FD_CUDA(cudaFuncSetAttribute(nms_cta_kernel<MODE, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        nms_cta_kernel<MODE, 0><<<B, NT, smem, ctx->stream>>>(a);
    }
    FD_LAUNCH_CHECK_NAMED(ctx, "nms_cta_kernel");
    if (dbg_on) {
        std::vector<long long> h(16 * (size_t)std::min(B, 4096));
        cudaStreamSynchronize(ctx->stream);
        cudaMemcpy(h.data(), dbg_dev, sizeof(long long) * h.size(), cudaMemcpyDeviceToHost);
        long long t0 = h[0];
        for (int b = 0; b < std::min(B, 4096); ++b) t0 = std::min(t0, h[16 * b]);
        for (int b = 0; b < std::min(B, 4096); ++b) {
            const long long *d = &h[16 * b];
            fprintf(stderr, "[nms dbg] cta %3d K=%4lld kept=%3lld iters=%2lld start+%6.2f load %5.2f sort %5.2f gather %5.2f greedy %6.2f us\n", b, d[6], d[7], d[5],
                    (d[0] - t0) * 1e-3, (d[1] - d[0]) * 1e-3, (d[2] - d[1]) * 1e-3, (d[3] - d[2]) * 1e-3, (d[4] - d[3]) * 1e-3);
        }
    }
    return FD_OK;
}

// One problem of SINGLE_PROBLEM_CROSSOVER < K <= MID_CAP boxes: a single cooperative launch (nms_mid_kernel).
static int nms_mid_impl(fd_ctx *ctx, const float *boxes, int K, int stride, const IouParams &iou, int mode, bool presorted, int32_t *keep_dev,
                        int32_t *num_keep_dev) {
    const int ntiles = (K + NT - 1) / NT;
    FD_TRY(ctx->nms_ws[1].reserve(sizeof(u64) * (size_t)K));
    FD_TRY(ctx->nms_ws[3].reserve(sizeof(float4) * (size_t)K));
    FD_TRY(ctx->nms_ws[5].reserve(sizeof(int) * (size_t)ntiles * 33 + 64));
    const size_t zero_ints = 32 + (size_t)K * 2 + ((size_t)K + 3) / 4;     // status block, list counters, ranks, decision states
    FD_TRY(ctx->nms_ws[6].reserve(sizeof(int) * zero_ints + 64));
    FD_TRY(ctx->nms_ws_sp[3].reserve(sizeof(int) * (size_t)K * ADJ_CAP));
    int *st = ctx->nms_ws[6].as<int>();
    int *adj_cnt = st + 32, *rank = adj_cnt + K;
    MidArgs m{};
    m.dets = boxes;
    m.n = K;
    m.stride = stride;
    m.presorted = presorted ? 1 : 0;
    m.mode = mode;
    m.sorted = ctx->nms_ws[1].as<u64>();
    m.sbox = ctx->nms_ws[3].as<float4>();
    m.rank = rank;
    m.st = st;
    m.zero_ints = (int)zero_ints;
    RoundsArgs &ra = m.ra;
    ra.N = K;
    ra.keys = m.sorted;
    ra.adj = ctx->nms_ws_sp[3].as<int>();
    ra.adj_cnt = adj_cnt;
    ra.state = reinterpret_cast<unsigned char *>(rank + K);
    ra.counters = st + 13;
    ra.tile_counts = ctx->nms_ws[5].as<int>();
    ra.ballots = reinterpret_cast<unsigned *>(ra.tile_counts + ntiles);
    ra.out_state = st + 3;
    ra.iou = iou;
    ra.sbox = m.sbox;
    ra.mode = mode;
    ra.status = st;
    ra.final_keep = keep_dev;
    ra.final_num = num_keep_dev;
    static int per_sm = 0;                                                 // one device type per process
    const size_t smem = sizeof(int) * (size_t)ADJ_SMEM * NT;
    if (!per_sm) {
        FD_CUDA(cudaFuncSetAttribute(nms_mid_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        FD_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, nms_mid_kernel, NT, smem));
        if (per_sm < 1) return fail(FD_ERR_CUDA, "nms_mid_kernel does not fit on an SM");
    }
    const int grid = ctx->num_sms * per_sm;
    m.slices = std::max(1, std::min((2 * grid + ntiles - 1) / ntiles, (K + 127) / 128));
    m.per_slice = (((K + m.slices - 1) / m.slices) + 1) & ~1;
    m.slices = (K + m.per_slice - 1) / m.per_slice;
    static const bool dbg_on = getenv("FD_NMS_DBG") != nullptr;             // phase timeline of block 0 on stderr
    static long long *dbg_dev = nullptr;
    if (dbg_on && !dbg_dev) FD_CUDA(cudaMalloc(&dbg_dev, sizeof(long long) * 16));
    ra.dbg = dbg_on ? dbg_dev : nullptr;
    void *args[] = {&m};
    FD_CUDA(cudaLaunchCooperativeKernel((const void *)nms_mid_kernel, dim3(grid), dim3(NT), args, smem, ctx->stream));
    FD_LAUNCH_CHECK_NAMED(ctx, "nms_mid_kernel");
    if (dbg_on) {
        long long h[8];
        int sth[8];
        cudaStreamSynchronize(ctx->stream);
        cudaMemcpy(h, dbg_dev, sizeof(h), cudaMemcpyDeviceToHost);
        cudaMemcpy(sth, st, sizeof(sth), cudaMemcpyDeviceToHost);
        fprintf(stderr, "[nms mid dbg] K=%d grid=%d slices=%d: zero %.1f  rank %.1f  scatter %.1f  lists %.1f  sweeps %.1f (epochs %d)  output %.1f us\n", K, grid,
                m.slices, (h[1] - h[0]) * 1e-3, (h[2] - h[1]) * 1e-3, (h[3] - h[2]) * 1e-3, (h[4] - h[3]) * 1e-3, (h[5] - h[4]) * 1e-3, sth[6],
                (h[6] - h[5]) * 1e-3);
    }
    return FD_OK;
}

// The big path as ONE cooperative launch (nms_big_kernel).  keys_in: optional keys (score desc | box index) in any order, else made
// from column 4 of boxes; box indices are below index_bound.  keep_count receives the count, nan_flag (optional) the NaN flag.
static int nms_big_one_launch(fd_ctx *ctx, const u64 *keys_in, const float *boxes, int K, int stride, int index_bound, float thr, int mode,
                              bool presorted, int32_t *keep_dev, int32_t *keep_count, int32_t *nan_flag) {
    const int ntiles = (K + NT - 1) / NT;
    FD_TRY(ctx->nms_ws[0].reserve(sizeof(u64) * (size_t)K));
    FD_TRY(ctx->nms_ws[1].reserve(sizeof(u64) * (size_t)K));
    FD_TRY(ctx->nms_ws[2].reserve(sizeof(int) * ((size_t)2 * CS_D * ntiles + CS_D)));
    FD_TRY(ctx->nms_ws[3].reserve(sizeof(float4) * (size_t)K));
    FD_TRY(ctx->nms_ws[4].reserve(sizeof(int) * (size_t)K * 3));
    FD_TRY(ctx->nms_ws[5].reserve(sizeof(float4) * HEAD + sizeof(int) * (size_t)ntiles * 33 + 64));
    FD_TRY(ctx->nms_ws[6].reserve(sizeof(int) * 32));
    FD_TRY(ctx->nms_ws_sp[0].reserve(sizeof(u64) * (size_t)K * 2));
    FD_TRY(ctx->nms_ws_sp[1].reserve(sizeof(int) * (size_t)(GRID_MAX_CELLS + 1) * 3));                                       // cell counts, starts, ends
    FD_TRY(ctx->nms_ws_sp[2].reserve((sizeof(float4) + sizeof(float) + sizeof(int) * 4) * (size_t)K + (size_t)K + 16));   // cbox, carea, tmp cell, 3 counters, state
    FD_TRY(ctx->nms_ws_sp[3].reserve(sizeof(int) * (size_t)K * ADJ_ROW3));
    int *st = ctx->nms_ws[6].as<int>();
    FD_CUDA(cudaMemsetAsync(st, 0, sizeof(int) * 32, ctx->stream));
    const IouParams iou = make_iou_params(thr, mode);
    BigArgs m{};
    m.dets = boxes;
    m.n = K;
    m.stride = stride;
    m.presorted = presorted ? 1 : 0;
    m.mode = mode;
    m.keys_in = keys_in;
    m.ibits = index_bound > 1 ? 32 - __builtin_clz((unsigned)(index_bound - 1)) : 0;
    m.key_e = ctx->nms_ws[0].as<u64>();
    m.tmp_key = ctx->nms_ws[1].as<u64>();
    m.ckey = ctx->nms_ws_sp[0].as<u64>();
    m.kept_keys = m.ckey + K;
    m.hist = ctx->nms_ws[2].as<int>();
    m.sbox = ctx->nms_ws[3].as<float4>();
    m.st = st;
    m.cell_cnt = ctx->nms_ws_sp[1].as<int>();
    m.cell_start = m.cell_cnt + (GRID_MAX_CELLS + 1);
    m.cell_end = m.cell_start + (GRID_MAX_CELLS + 1);
    m.cbox = ctx->nms_ws_sp[2].as<float4>();
    m.carea = reinterpret_cast<float *>(m.cbox + K);
    m.tmp_cell = reinterpret_cast<int *>(m.carea + K);
    int *adj_cnt = m.tmp_cell + K;
    float4 *ks = ctx->nms_ws[5].as<float4>();
    int *tile_counts = reinterpret_cast<int *>(ks + HEAD);
    unsigned *ballots = reinterpret_cast<unsigned *>(tile_counts + ntiles);
    int *stream_a = ctx->nms_ws[4].as<int>(), *stream_b = stream_a + K, *keep_ranks = stream_b + K;
    m.cell_e = stream_a;        // (the peel's streams and kept ranks: the grid path and the peel exclude each other)
    m.slot_e = stream_b;
    m.kept_rank = keep_ranks;
    RoundsArgs &ra = m.ra;
    ra.N = K;
    ra.keys = m.ckey;
    ra.cell_start = m.cell_start;
    ra.cell_end = m.cell_end;
    ra.cbox = m.cbox;
    ra.carea = m.carea;
    ra.adj = ctx->nms_ws_sp[3].as<int>();
    ra.adj_cnt = adj_cnt;
    ra.state = reinterpret_cast<unsigned char *>(adj_cnt + (size_t)3 * K);
    ra.counters = st + 13;
    ra.tile_counts = tile_counts;
    ra.ballots = ballots;
    ra.out_state = st + 3;
    ra.iou = iou;
    ra.kept_keys = m.kept_keys;
    PeelArgs &pa = m.pa;
    pa.sbox = m.sbox;
    pa.N = K;
    pa.stream_a = stream_a;
    pa.stream_b = stream_b;
    pa.keep_ranks = keep_ranks;
    pa.state = st + 3;
    pa.ks = ks;
    pa.tile_counts = tile_counts;
    pa.ballots = ballots;
    pa.status = st;
    pa.iou = iou;
    m.keep_dev = keep_dev;
    m.keep_count = keep_count;
    m.nan_flag = nan_flag;
    static int per_sm = 0;                                                 // one device type per process
    const size_t smem = std::max(std::max(sizeof(int) * (size_t)ADJ_SMEM * NT, sizeof(PeelSmem)), CS_SMEM);
    if (!per_sm) {
        FD_CUDA(cudaFuncSetAttribute(nms_big_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        FD_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, nms_big_kernel, NT, smem));
        if (per_sm < 1) return fail(FD_ERR_CUDA, "nms_big_kernel does not fit on an SM");
    }
    static const bool dbg_on = getenv("FD_NMS_DBG") != nullptr;             // phase timeline of block 0 on stderr
    static long long *dbg_dev = nullptr;
    if (dbg_on && !dbg_dev) FD_CUDA(cudaMalloc(&dbg_dev, sizeof(long long) * 16));
    m.dbg = dbg_on ? dbg_dev : nullptr;
    void *args[] = {&m};
    FD_CUDA(cudaLaunchCooperativeKernel((const void *)nms_big_kernel, dim3(ctx->num_sms * per_sm), dim3(NT), args, smem, ctx->stream));
    FD_LAUNCH_CHECK_NAMED(ctx, "nms_big_kernel");
    if (dbg_on) {
        long long h[16];
        int sth[32];
        cudaStreamSynchronize(ctx->stream);
        cudaMemcpy(h, dbg_dev, sizeof(h), cudaMemcpyDeviceToHost);
        cudaMemcpy(sth, st, sizeof(sth), cudaMemcpyDeviceToHost);
        fprintf(stderr, "[nms big dbg] K=%d grid=%d spatial=%d: keys+stats %.1f  cells %.1f  scan %.1f  scatter %.1f  order %.1f  lists %.1f  sweeps %.1f (lists loaded by %.1f, first epoch's sweeps until %.1f)  kept order %.1f (epochs %d, list refills %d) us, total %.1f\n",
                K, ctx->num_sms * per_sm, sth[3], (h[1] - h[0]) * 1e-3, (h[2] - h[1]) * 1e-3, (h[3] - h[2]) * 1e-3, (h[4] - h[3]) * 1e-3,
                (h[5] - h[4]) * 1e-3, (h[6] - h[5]) * 1e-3, (h[9] - h[6]) * 1e-3, (h[11] - h[6]) * 1e-3, (h[12] - h[6]) * 1e-3, (h[8] - h[7]) * 1e-3, sth[6], sth[7],
                (h[8] - h[0]) * 1e-3);
    }
    return FD_OK;
}

// Statistics of the last big-path NMS: [0] spatial path used, [1] kept, [2] decision epochs, [3] grid w, [4] grid h,
// [5] cell size (float bits)
int nms_last_stats(fd_ctx *ctx, int32_t out[8]) {
    for (int i = 0; i < 8; ++i) out[i] = 0;
    if (!ctx->nms_ws[6].p) return FD_OK;
    int st[32];
    FD_CUDA(cudaMemcpyAsync(st, ctx->nms_ws[6].p, sizeof(st), cudaMemcpyDeviceToHost, ctx->stream));
    FD_CUDA(cudaStreamSynchronize(ctx->stream));
    out[0] = st[3]; out[1] = st[4]; out[2] = st[6]; out[3] = st[19]; out[4] = st[20]; out[5] = st[18];
    return FD_OK;
}

// Generic device NMS on a (K, stride) row-major array with the score in column 4 (ignored if presorted).
// keep_dev (K) and num_keep_dev (2 ints: [0] count, [1] NaN flag) are device buffers.
constexpr int SINGLE_PROBLEM_CROSSOVER = 1024;   // = TINY_CAP: beyond it the all-SM mid path is faster (61 vs 68 us at 1 100 boxes)
int nms_device(fd_ctx *ctx, const float *dets_dev, int K, int stride, float thr, int mode, bool presorted,
               int32_t *keep_dev, int32_t *num_keep_dev) {
    // ONE problem: a single SM (the barrier-light tiny path) up to 1 024 boxes, one cooperative all-SM kernel up to MID_CAP,
    // nms_big_kernel beyond (measured: profiles/r2_nms_sizes.json); batched callers keep one CTA per image up to SMALL_CAP
    static const int single_cross = getenv("FD_NMS_CROSS") ? atoi(getenv("FD_NMS_CROSS")) : SINGLE_PROBLEM_CROSSOVER;
    static const int mid_cap = getenv("FD_NMS_MID_CAP") ? atoi(getenv("FD_NMS_MID_CAP")) : MID_CAP;   // 0: A/B without the mid path
    if (K > std::min(SMALL_CAP, single_cross) && K <= mid_cap)
        return nms_mid_impl(ctx, dets_dev, K, stride, make_iou_params(thr, mode), mode, presorted, keep_dev, num_keep_dev);
    FD_TRY(ctx->nms_ws[7].reserve(sizeof(int) * 8));
    int *status = ctx->nms_ws[7].as<int>();
    FD_CUDA(cudaMemsetAsync(status, 0, sizeof(int) * 8, ctx->stream));
    if (K <= std::min(SMALL_CAP, single_cross)) {
        SmallArgs a{};
        a.keys = nullptr;
        a.key_stride = 0;
        a.boxes = dets_dev;
        a.box_batch_stride = 0;
        a.box_stride = stride;
        a.counts = nullptr;
        a.K = K;
        a.presorted = presorted ? 1 : 0;
        a.sort_only = 0;
        a.iou = make_iou_params(thr, mode);
        a.keep = keep_dev;
        a.keep_stride = 0;
        a.keep_count = num_keep_dev;
        a.status = status;
        a.big_list = nullptr;
        if (presorted) {
            // presorted rows carry no usable score column contract (boxes_dim may be 4): keys = identity
            FD_TRY(ctx->nms_ws[0].reserve(sizeof(u64) * (size_t)std::max(K, 1)));
            iota_keys_kernel<<<(K + 255) / 256, 256, 0, ctx->stream>>>(K, ctx->nms_ws[0].as<u64>());
            FD_LAUNCH_CHECK(ctx);
            a.keys = ctx->nms_ws[0].as<u64>();
        }
        if (mode == 0) FD_TRY(launch_small<0>(ctx, a, 1, false));
        else FD_TRY(launch_small<1>(ctx, a, 1, false));
        FD_CUDA(cudaMemcpyAsync(num_keep_dev + 1, status, sizeof(int), cudaMemcpyDeviceToDevice, ctx->stream));
        return FD_OK;
    }
    return nms_big_one_launch(ctx, nullptr, dets_dev, K, stride, K, thr, mode, presorted, keep_dev, num_keep_dev, num_keep_dev + 1);
}

// argsort_descending on the device: order_dev (n), flag_dev (1 int: NaN flag)
int argsort_device(fd_ctx *ctx, const float *scores_as_dets, int n, int stride, int32_t *order_dev, int32_t *flag_dev) {
    FD_TRY(ctx->nms_ws[7].reserve(sizeof(int) * 8));
    int *status = ctx->nms_ws[7].as<int>();
    FD_CUDA(cudaMemsetAsync(status, 0, sizeof(int) * 8, ctx->stream));
    if (n <= SMALL_CAP) {
        SmallArgs a{};
        a.boxes = scores_as_dets;  // score read at column 4 -> caller passes (scores - 4) with stride 1
        a.box_stride = stride;
        a.K = n;
        a.sort_only = 1;
        a.keep = order_dev;
        a.keep_count = status + 4;
        a.status = status;
        FD_TRY(launch_small<0>(ctx, a, 1, false));
        FD_CUDA(cudaMemcpyAsync(flag_dev, status, sizeof(int), cudaMemcpyDeviceToDevice, ctx->stream));
        return FD_OK;
    }
    const int ntiles = (n + NT - 1) / NT;
    FD_TRY(ctx->nms_ws[0].reserve(sizeof(u64) * (size_t)n));
    FD_TRY(ctx->nms_ws[1].reserve(sizeof(u64) * (size_t)n));
    FD_TRY(ctx->nms_ws[2].reserve(sizeof(int) * ((size_t)2 * CS_D * ntiles + CS_D)));
    u64 *keys = ctx->nms_ws[0].as<u64>(), *tmp = ctx->nms_ws[1].as<u64>();
    int *hist = ctx->nms_ws[2].as<int>();
    static int per_sm = 0;                                                 // one device type per process
    if (!per_sm) {
        FD_CUDA(cudaFuncSetAttribute(argsort_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CS_SMEM));
        FD_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, argsort_kernel, NT, CS_SMEM));
        if (per_sm < 1) return fail(FD_ERR_CUDA, "argsort_kernel does not fit on an SM");
    }
    const int grid = std::min(ctx->num_sms * per_sm, ntiles);             // every CTA owns at least one tile
    void *args[] = {(void *)&scores_as_dets, &n, &stride, &keys, &tmp, &hist, &status, &order_dev, &flag_dev};
    FD_CUDA(cudaLaunchCooperativeKernel((const void *)argsort_kernel, dim3(grid), dim3(NT), args, CS_SMEM, ctx->stream));
    FD_LAUNCH_CHECK_NAMED(ctx, "argsort_kernel");
    return FD_OK;
}

// Batched: one CTA per image over the decode kernel's candidate buffers.
int nms_batch_launch(fd_ctx *ctx, int B, float iou_thr) {
    const int TA = ctx->dcfg.total_anchors;
    SmallArgs a{};
    a.keys = ctx->cand_keys.as<u64>();
    a.key_stride = (size_t)TA;
    a.boxes = ctx->cand_box.as<float>();
    a.box_batch_stride = (size_t)TA * 4;
    a.box_stride = 4;
    a.counts = ctx->cand_count.as<int>();
    a.K = 0;
    a.presorted = 0;
    a.sort_only = 0;
    a.iou = make_iou_params(iou_thr, 0);
    a.keep = ctx->keep_src.as<int>();
    a.keep_stride = (size_t)TA;
    a.keep_count = ctx->keep_count.as<int>();
    a.status = ctx->status();
    a.big_list = ctx->big_list.as<int>();
    return launch_small<0>(ctx, a, B, true);
}

// General single-CTA path for ONE image of the batch (1024 < K <= SMALL_CAP after the fused kernel deferred it).
int nms_batch_small_image(fd_ctx *ctx, int b, int K, float iou_thr) {
    const int TA = ctx->dcfg.total_anchors;
    SmallArgs a{};
    a.keys = ctx->cand_keys.as<u64>() + (size_t)b * TA;
    a.key_stride = (size_t)TA;
    a.boxes = ctx->cand_box.as<float>() + (size_t)b * TA * 4;
    a.box_batch_stride = (size_t)TA * 4;
    a.box_stride = 4;
    a.counts = nullptr;
    a.K = K;
    a.iou = make_iou_params(iou_thr, 0);
    a.keep = ctx->keep_src.as<int>() + (size_t)b * TA;
    a.keep_stride = (size_t)TA;
    a.keep_count = ctx->keep_count.as<int>() + b;
    a.status = ctx->status() + 4;   // scratch flags: the batch's own flags were already read
    a.big_list = nullptr;
    return launch_small<0>(ctx, a, 1, true);
}

// Big path for one image of the batch (K > SMALL_CAP): nms_big_kernel on the decode kernel's keys, which are in slot (compaction)
// order and carry anchor ids up to the total anchor count; boxes are float4 by anchor id.
int nms_batch_big_image(fd_ctx *ctx, int b, int K, float iou_thr) {
    const int TA = ctx->dcfg.total_anchors;
    return nms_big_one_launch(ctx, ctx->cand_keys.as<u64>() + (size_t)b * TA, ctx->cand_box.as<float>() + (size_t)b * TA * 4, K, 4, TA,
                              iou_thr, 0, false, ctx->keep_src.as<int>() + (size_t)b * TA, ctx->keep_count.as<int>() + b, nullptr);
}

}  // namespace fd
