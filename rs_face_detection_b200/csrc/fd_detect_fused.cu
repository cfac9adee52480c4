// fd_detect_fused.cu — the whole post-CNN half of RetinaFaceDetection::_forward + _postprocess (face_detection.rs:319-493)
// and the similarity estimate of FaceAlignment::call (face_alignment.rs:50-59) in ONE kernel launch, one CTA per image:
//
//   score scan      the 2A foreground score planes of the image, 128-bit loads, `>= conf_thr` (face_detection.rs:374-379),
//                   warp-aggregated compaction of sort keys (score desc | anchor id) into shared memory;
//   head fetch      as soon as the keys are compacted, every candidate's box deltas, landmark deltas and score are copied
//                   into shared memory (cp.async), in flight during the sort; decode and gather read them from there;
//   sort            rank sort: keys are unique, so a key's rank is the number of smaller keys — sorted runs of 32 per warp,
//                   then binary searches of the other runs; ascending keys == the reference's stable descending sort over
//                   the 32|16|8 concatenation (utils.rs:87-95, face_detection.rs:410-430);
//   decode          bbox_pred + clip_boxes for the candidates only, scattered to their sorted rank;
//   NMS             exact greedy (nms.rs:3-65) in shared memory / registers (fd_nms_tiny.cuh);
//   offsets         every CTA publishes its kept count (epoch-tagged) and sums its predecessors' — no chain, no second launch;
//   gather          kept boxes / landmark_pred / `÷ det_scale` (face_detection.rs:432-493) straight to the compact outputs;
//   estimate        LMedS similarity per kept face, 16 lanes each (fd_estimate.cuh), for the warp kernel that follows.
//
// Per-image candidate lists longer than 1024 (conf_thr far below the reference's 0.7, or ~50 faces per frame) are decoded to
// the global candidate buffers; up to 4096 candidates the same CTA runs the general single-CTA NMS (fd_nms_small.cuh) in
// place once the ctx has met such an image (the launch then reserves that path's shared memory); otherwise, and always
// beyond 4096, the image is deferred and fd_detect_fetch completes it with the general NMS paths of fd_nms.cu.
// The three-kernel path (decode_kernel, nms_cta_kernel, finalize_kernel) remains for geometries without 128-bit score rows
// and as the A/B reference (FD_NO_FUSED=1).
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <vector>
#include "fd_internal.cuh"
#include "fd_decode.cuh"
#include "fd_nms_tiny.cuh"
#include "fd_nms_small.cuh"
#include "fd_estimate.cuh"

namespace fd {

constexpr int FT = 1024;
constexpr int FUSED_DBG_IMAGES = 4096;   // FD_FUSED_DBG=1 timestamps are kept for the first 4096 images of a launch

struct FusedArgs {
    DecodeCfg c;
    HeadPtrs hp;
    float conf_thr;
    IouParams iou;
    u64 *keys;            // [B][TA] candidate keys (global copy, read by the deferred paths)
    float4 *cand_box;     // [B][TA] by anchor id (kept boxes always; every candidate of a deferred image)
    float *cand_rec;      // [B][TA][12]
    int *counts;          // [B] candidates per image
    int *keep;            // [B][TA] kept anchor ids in pick order
    int *keep_count;      // [B]  (-1: deferred)
    int *status;          // [0] unused, [1] deferred images, [2] total faces
    int *status_next;     // the other half of the ping-pong: zeroed by the last CTA for the next call
    int *big_list;
    const float *det_scale;
    int *offsets;         // [B+1]
    float *out_det;       // [total][5]
    float *out_lmk;       // [total][10]
    int *out_frame_idx;   // [total]
    EstConst ec;
    double *M12;          // [est_cap][12]
    uint8_t *ok;          // [est_cap]
    int est_cap;
    int *ticket;          // [0] next image, [1] CTAs finished (both zero between launches)
    u64 *agg;             // [B] (epoch << 32) | kept count
    unsigned epoch;
    int B;
    int general_ok;       // the dynamic shared memory has room for the general single-CTA NMS (1024 < K <= 4096 on the device)
    long long *dbg;       // FD_FUSED_DBG=1: per-CTA stage timestamps
};

// Shared memory of one image's CTA: a small control block, then a work area that is either the K <= 1024 state below or,
// for an image with 1024 < K <= 4096 candidates, the general path's SmallSmem (fd_nms_small.cuh) — the launch reserves room
// for that only when the ctx has seen such images (`general_ok`); the rows of the kept faces (flmk / fdet) are written after
// the NMS, when either state is dead.
struct FusedCtrl {
    int red[33];
    int b, cnt, kept, off, general;
};
constexpr int FUSED_CTRL_BYTES = 256;
static_assert(sizeof(FusedCtrl) <= FUSED_CTRL_BYTES, "control block");
struct FusedSmem {
    TinySmem t;
    u64 ckey[TINY_CAP];          // candidate keys in arrival order (slot)
    int rank[TINY_CAP];          // sorted rank of slot i
    int slot[TINY_CAP];          // slot of rank r
    union {
        float head[TINY_CAP][15];   // until the gather has read it: raw box deltas [0..3], landmark deltas [4..13], fg score [14] of slot i
        struct {
            float flmk[TINY_CAP * 10];   // rescaled landmarks of the kept faces (output rows, input of the estimate)
            float fdet[TINY_CAP * 5];    // rescaled boxes + score of the kept faces (output rows)
        };
    };
};
static_assert(FUSED_CTRL_BYTES + sizeof(FusedSmem) <= 227 * 1024, "fused detect shared memory");

__device__ __forceinline__ u64 ld_acquire_u64(const u64 *p) {
    u64 v;
    asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_u64(u64 *p, u64 v) {
    asm volatile("st.release.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ void cp_async4(float *dst_smem, const float *src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"((unsigned)__cvta_generic_to_shared(dst_smem)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }

// ascending bitonic network over the 32 keys of a warp; each key's slot moves with it
__device__ __forceinline__ void warp_sort_slots(u64 &key, int &slot, int lane) {
#pragma unroll
    for (int k = 2; k <= 32; k <<= 1) {
#pragma unroll
        for (int j = k >> 1; j > 0; j >>= 1) {
            const u64 okey = __shfl_xor_sync(0xffffffffu, key, j);
            const int oslot = __shfl_xor_sync(0xffffffffu, slot, j);
            const bool take_min = ((lane & j) == 0) == ((lane & k) == 0);
            if (take_min == (okey < key)) {
                key = okey;
                slot = oslot;
            }
        }
    }
}
// number of keys below `key` in an ascending run of 32
__device__ __forceinline__ int count_below(const u64 *run, u64 key) {
    int p = 0;
#pragma unroll
    for (int s = 16; s > 0; s >>= 1)
        if (run[p + s - 1] < key) p += s;
    return p + (run[p] < key ? 1 : 0);
}

// Score scan of image b: UN items (4 consecutive positions of one stride each) per thread are loaded before any is
// processed, so the image's 2A score planes (134 KB for 640x640) cost about one memory latency.  AT: compile-time A (0 = runtime).
template <int AT, int UN>
__device__ __forceinline__ void fused_score_scan(const FusedArgs &a, FusedSmem &sm, FusedCtrl &ctl, int b) {
    const DecodeCfg &c = a.c;
    constexpr int AMAX = AT ? AT : FD_MAX_ANCHORS;
    const int A = AT ? AT : c.A;
    const int tid = threadIdx.x, lane = tid & 31;
    const size_t img_base = (size_t)b * c.total_anchors;
    const int nq = c.total_pos >> 2;   // every H*W is a multiple of 4 (checked by the host)
    for (int q0 = 0; q0 < nq; q0 += UN * FT) {
        float4 v[UN][AMAX];
        int s_[UN], local_[UN];
        bool act[UN];
#pragma unroll
        for (int u = 0; u < UN; ++u) {
            const int q = q0 + u * FT + tid;
            act[u] = q < nq;
            const int pos = act[u] ? q * 4 : 0;
            s_[u] = stride_of_pos(c, pos);
            local_[u] = pos - c.pos_off[s_[u]];
            const int hw = c.fh[s_[u]] * c.fw[s_[u]];
            const float *sc = a.hp.p[3 * s_[u]] + (size_t)b * 2 * A * hw;
#pragma unroll
            for (int aa = 0; aa < AMAX; ++aa)   // fg scores are channels A.. (face_detection.rs:322)
                v[u][aa] = (act[u] && aa < A) ? __ldg(reinterpret_cast<const float4 *>(sc + (size_t)(A + aa) * hw + local_[u]))
                                              : make_float4(0.f, 0.f, 0.f, 0.f);
        }
#pragma unroll
        for (int u = 0; u < UN; ++u) {
            if (q0 + u * FT >= nq) break;   // uniform
            unsigned pass = 0;              // bit aa*4+k
            if (act[u]) {
#pragma unroll
                for (int aa = 0; aa < AMAX; ++aa) {
                    if (aa >= A) break;
                    const float sv4[4] = {v[u][aa].x, v[u][aa].y, v[u][aa].z, v[u][aa].w};
#pragma unroll
                    for (int k = 0; k < 4; ++k)   // face_detection.rs:375; a NaN score fails `>=` and is dropped like any low score
                        if (sv4[k] >= a.conf_thr) pass |= 1u << (aa * 4 + k);
                }
            }
            const int cnt = __popc(pass);
            if (__ballot_sync(0xffffffffu, cnt != 0) == 0) continue;   // common case: nothing above the threshold in this warp
            int incl = cnt;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int nb = __shfl_up_sync(0xffffffffu, incl, o);
                if (lane >= o) incl += nb;
            }
            int base = 0;
            if (lane == 31) base = atomicAdd(&ctl.cnt, incl);
            base = __shfl_sync(0xffffffffu, base, 31);
            int slot = base + incl - cnt;
            while (pass) {
                const int bit = __ffs(pass) - 1;
                pass &= pass - 1;
                const int aa = bit >> 2, k = bit & 3;
                float sv = 0.0f;
#pragma unroll
                for (int x = 0; x < AMAX; ++x) {
                    const float sv4[4] = {v[u][x].x, v[u][x].y, v[u][x].z, v[u][x].w};
#pragma unroll
                    for (int y = 0; y < 4; ++y)
                        if (x == aa && y == k) sv = sv4[y];
                }
                const int id = c.anchor_off[s_[u]] + (local_[u] + k) * A + aa;
                const u64 key = ((u64)desc_key(sv) << 32) | (unsigned)id;
                if (slot < TINY_CAP) sm.ckey[slot] = key;
                a.keys[img_base + slot] = key;
                ++slot;
            }
        }
    }
}

__device__ __forceinline__ void fused_stamp(const FusedArgs &a, int b, int slot) {
    if (a.dbg && threadIdx.x == 0 && b < FUSED_DBG_IMAGES) {
        long long t;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
        a.dbg[b * 16 + slot] = t;
    }
}

__device__ __forceinline__ void detect_fused_body(const FusedArgs &a) {
    extern __shared__ __align__(16) unsigned char fused_raw[];
    FusedCtrl &ctl = *reinterpret_cast<FusedCtrl *>(fused_raw);
    FusedSmem &sm = *reinterpret_cast<FusedSmem *>(fused_raw + FUSED_CTRL_BYTES);
    const DecodeCfg &c = a.c;
    const int tid = threadIdx.x, lane = tid & 31;
    pdl_trigger();   // the warp kernel's CTAs may take the SMs this grid leaves idle (they wait for its completion)
    if (tid == 0) {
        ctl.cnt = 0;
        ctl.kept = 0;
        ctl.general = 0;
    }
    sm.rank[tid] = 0;   // (FT == TINY_CAP)
    pdl_wait();
    if (tid == 0) ctl.b = atomicAdd(a.ticket, 1);   // images in ticket order: every predecessor of this image is already running
    __syncthreads();
    const int b = ctl.b;
    fused_stamp(a, b, 0);
    const int A = c.A, TA = c.total_anchors;
    const size_t img_base = (size_t)b * TA;

    // ---- 1. score scan + key compaction ----
    if (c.A == 2) fused_score_scan<2, 3>(a, sm, ctl, b);
    else fused_score_scan<0, 1>(a, sm, ctl, b);
    __syncthreads();
    fused_stamp(a, b, 1);
    const int K = ctl.cnt;
    if (tid == 0) a.counts[b] = K;
    if (K <= TINY_CAP && tid < K) {   // head fetch of slot tid: in flight during the sort, waited for by this thread only
        int s, local, aa;
        split_anchor_id(c, (int)(unsigned)sm.ckey[tid], s, local, aa);
        const int hw = c.fh[s] * c.fw[s];
        const float *bb = a.hp.p[3 * s + 1] + (size_t)b * 4 * A * hw + local;
        const float *lm = a.hp.p[3 * s + 2] + (size_t)b * 10 * A * hw + local;
        float *dst = sm.head[tid];
#pragma unroll
        for (int k = 0; k < 4; ++k) cp_async4(dst + k, bb + (size_t)(4 * aa + k) * hw);
#pragma unroll
        for (int k = 0; k < 10; ++k) cp_async4(dst + 4 + k, lm + (size_t)(10 * aa + k) * hw);
        cp_async4(dst + 14, a.hp.p[3 * s] + (size_t)b * 2 * A * hw + (size_t)(A + aa) * hw + local);
    }

    // ---- 2. sort + decode + NMS (K <= 1024), or decode everything and defer ----
    int *keep = a.keep + img_base;
    if (K > TINY_CAP) {
        for (int i = tid; i < K; i += FT) {
            const int id = (int)(unsigned)a.keys[img_base + i];
            int s, local, aa;
            split_anchor_id(c, id, s, local, aa);
            const AnchorGeo g = anchor_geo(c, s, local, aa);
            a.cand_box[img_base + id] = decode_box(c, a.hp, b, s, local, aa, g);
            float rec[CAND_REC];
            decode_landmarks(c, a.hp, b, s, local, aa, g, rec);
            const int hw = c.fh[s] * c.fw[s];
            rec[10] = __ldg(a.hp.p[3 * s] + (size_t)b * 2 * A * hw + (size_t)(A + aa) * hw + local);
            rec[11] = 0.0f;
            float4 *dst = reinterpret_cast<float4 *>(a.cand_rec + (img_base + id) * CAND_REC);
            dst[0] = make_float4(rec[0], rec[1], rec[2], rec[3]);
            dst[1] = make_float4(rec[4], rec[5], rec[6], rec[7]);
            dst[2] = make_float4(rec[8], rec[9], rec[10], rec[11]);
        }
        bool handled = false;
        if (a.general_ok && K <= SMALL_CAP) {   // the general single-CTA path, in place of the K <= 1024 one
            __syncthreads();                     // keys and boxes of this image are in global memory: visible to the block
            SmallArgs sa{};
            sa.keys = a.keys;
            sa.key_stride = (size_t)TA;
            sa.boxes = reinterpret_cast<const float *>(a.cand_box);
            sa.box_batch_stride = (size_t)TA * 4;
            sa.box_stride = 4;
            sa.K = K;
            sa.iou = a.iou;
            sa.keep = a.keep;
            sa.keep_stride = (size_t)TA;
            sa.keep_count = a.keep_count;
            sa.status = a.status;
            nms_general_cta<0, 4>(sa, *reinterpret_cast<SmallSmem *>(fused_raw + FUSED_CTRL_BYTES), b, K);
            __syncthreads();
            const int nk = a.keep_count[b];      // written by thread 0 of this CTA before the barrier
            if (nk >= 0 && nk <= TINY_CAP) {     // (more kept faces than the row staging holds: leave it to the host path)
                handled = true;
                if (tid == 0) {
                    ctl.kept = nk;
                    ctl.general = 1;
                }
            }
        }
        if (!handled && tid == 0) {
            a.keep_count[b] = -1;
            a.big_list[atomicAdd(&a.status[1], 1)] = b;
        }
    } else if (K > 0) {
        int n2 = 32;
        while (n2 < K) n2 <<= 1;
        {   // rank of slot i.  Every warp sorts the keys of its 32 slots (shuffle network, carrying the slot) into a run; a key's
            // rank is its place in its run plus, for every other run, the number of that run's keys below it (binary search).
            // The FT / (32 runs) parts of the block take every parts-th run each.
            const int nruns = (K + 31) >> 5, ne = nruns * 32, parts = FT / ne;
            u64 *run_key = sm.t.xch[0], *run_slot = sm.t.xch[1];
            if (tid < ne) {
                u64 key = tid < K ? sm.ckey[tid] : ~0ull;
                int slot = tid;
                warp_sort_slots(key, slot, lane);
                run_key[tid] = key;
                run_slot[tid] = (u64)slot;
            }
            __syncthreads();
            const int part = tid / ne, e = tid - part * ne;
            if (part < parts && run_key[e] != ~0ull) {
                const u64 key = run_key[e];
                const int w = e >> 5;
                int cnt = part == 0 ? (e & 31) : 0;
#pragma unroll 4
                for (int r = part; r < nruns; r += parts)
                    if (r != w) cnt += count_below(run_key + 32 * r, key);
                const int slot = (int)run_slot[e];
                if (parts == 1) sm.rank[slot] = cnt;
                else atomicAdd(&sm.rank[slot], cnt);
            }
        }
        __syncthreads();
        fused_stamp(a, b, 2);
        bool ok = true;
        if (tid < K) {   // decode slot tid into rank order
            const int r = sm.rank[tid], id = (int)(unsigned)sm.ckey[tid];
            int s, local, aa;
            split_anchor_id(c, id, s, local, aa);
            cp_async_wait_all();
            const float4 bx = decode_box(c, sm.head[tid], anchor_geo(c, s, local, aa));
            sm.t.sbox[r] = bx;
            sm.t.sarea[r] = box_area(bx);
            sm.t.sidx[r] = id;
            sm.slot[r] = tid;
            ok = box_is_fast_ok(bx);
        }
        const bool fast = !__syncthreads_or(!ok) && a.iou.fast;   // also publishes sbox / sidx / slot
        fused_stamp(a, b, 3);
        if (tid < n2) {   // whole warps; their barriers are named barrier 2 over n2 threads
            const float4 my = tid < K ? sm.t.sbox[tid] : make_float4(0.f, 0.f, 0.f, 0.f);
            const int nk = fast ? tiny_greedy<0, true>(sm.t, a.iou, K, n2, keep, my, nullptr)
                                : tiny_greedy<0, false>(sm.t, a.iou, K, n2, keep, my, nullptr);
            if (tid == 0) {
                ctl.kept = nk;
                a.keep_count[b] = nk;
            }
        }
    } else if (tid == 0) {
        a.keep_count[b] = 0;
    }
    __syncthreads();
    const int M = ctl.kept;
    const bool general = ctl.general != 0;
    fused_stamp(a, b, 4);

    // ---- 3. publish this image's kept count (epoch-tagged); the predecessors' counts are summed in step 5 ----
    if (tid == 0) st_release_u64(a.agg + b, ((u64)a.epoch << 32) | (unsigned)M);

    // ---- 4. gather + rescale (division, face_detection.rs:477-483) into shared memory: needs no offset yet ----
    const float ds = a.det_scale[b];
    float4 bx;
    float rec[CAND_REC];
    const int m = tid;   // M <= TINY_CAP == FT: one kept face per thread at most
    if (m < M) {
        if (general) {   // kept anchor ids from the general path; boxes / landmarks / score were decoded to global memory
            const int id = keep[m];
            bx = a.cand_box[img_base + id];
            const float4 *src = reinterpret_cast<const float4 *>(a.cand_rec + (img_base + id) * CAND_REC);
            const float4 r0 = src[0], r1 = src[1], r2 = src[2];
            rec[0] = r0.x; rec[1] = r0.y; rec[2] = r0.z; rec[3] = r0.w; rec[4] = r1.x; rec[5] = r1.y; rec[6] = r1.z; rec[7] = r1.w;
            rec[8] = r2.x; rec[9] = r2.y; rec[10] = r2.z; rec[11] = r2.w;
        } else {
            const int rank = sm.t.krank[m];
            const int id = sm.t.sidx[rank];
            const float *raw = sm.head[sm.slot[rank]];
            bx = sm.t.sbox[rank];
            int s, local, aa;
            split_anchor_id(c, id, s, local, aa);
            decode_landmarks(c, raw + 4, anchor_geo(c, s, local, aa), rec);
            rec[10] = raw[14];
            rec[11] = 0.0f;
            a.cand_box[img_base + id] = bx;   // the lazily-run general finalize reads these for every image of the batch
            float4 *dst = reinterpret_cast<float4 *>(a.cand_rec + (img_base + id) * CAND_REC);
            dst[0] = make_float4(rec[0], rec[1], rec[2], rec[3]);
            dst[1] = make_float4(rec[4], rec[5], rec[6], rec[7]);
            dst[2] = make_float4(rec[8], rec[9], rec[10], rec[11]);
        }
    }
    __syncthreads();   // every kept face's head values are read: fdet / flmk may overwrite them
    if (m < M) {
        float *d = sm.fdet + m * 5;
        d[0] = __fdiv_rn(bx.x, ds);
        d[1] = __fdiv_rn(bx.y, ds);
        d[2] = __fdiv_rn(bx.z, ds);
        d[3] = __fdiv_rn(bx.w, ds);
        d[4] = rec[10];
#pragma unroll
        for (int k = 0; k < 10; ++k) sm.flmk[m * 10 + k] = __fdiv_rn(rec[k], ds);
    }
    __syncthreads();
    fused_stamp(a, b, 5);

    // ---- 5. similarity estimate per kept face (for the warp kernel of fd_align_detections).  The first pass is computed
    //         BEFORE the wait for the predecessors' counts, so the estimate hides behind the slowest image of the batch;
    //         the compact outputs are written as soon as the offset is known. ----
    int off = 0;
    for (int f0 = 0; f0 == 0 || f0 < M; f0 += FT / EST_LANES) {
        const int f = f0 + tid / EST_LANES, sub = tid % EST_LANES;
        const bool live = f < M;
        float from[10], to[10];
#pragma unroll
        for (int k = 0; k < 10; ++k) {
            from[k] = live ? sm.flmk[f * 10 + k] : 0.0f;
            to[k] = a.ec.tmpl[k];
        }
        double Mx[6], iM[6];
        bool ok;
        estimate_group(a.ec, from, to, live, sub, Mx, iM, ok);
        if (f0 == 0) {
            fused_stamp(a, b, 6);
            int part = 0;   // every predecessor holds an earlier ticket, i.e. is running or done: the spin cannot deadlock
            for (int i = tid; i < b; i += FT) {
                u64 v = ld_acquire_u64(a.agg + i);
                while ((unsigned)(v >> 32) != a.epoch) {
                    __nanosleep(64);
                    v = ld_acquire_u64(a.agg + i);
                }
                part += (int)(unsigned)v;
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
            if (lane == 0) ctl.red[tid >> 5] = part;
            __syncthreads();
#pragma unroll
            for (int k = 0; k < FT / 32; ++k) off += ctl.red[k];
            if (tid == 0) {
                a.offsets[b] = off;
                if (b == a.B - 1) {
                    a.offsets[a.B] = off + M;
                    a.status[2] = off + M;
                }
            }
            for (int i = tid; i < M * 5; i += FT) a.out_det[(size_t)off * 5 + i] = sm.fdet[i];
            for (int i = tid; i < M * 10; i += FT) a.out_lmk[(size_t)off * 10 + i] = sm.flmk[i];
            for (int m = tid; m < M; m += FT) a.out_frame_idx[off + m] = b;
        }
        if (live && sub == 0 && off + f < a.est_cap) {
#pragma unroll
            for (int k = 0; k < 6; ++k) {
                a.M12[(size_t)(off + f) * 12 + k] = Mx[k];
                a.M12[(size_t)(off + f) * 12 + 6 + k] = iM[k];
            }
            a.ok[off + f] = ok ? 1 : 0;
        }
    }

    __syncthreads();
    fused_stamp(a, b, 7);
    if (a.dbg && tid == 0 && b < FUSED_DBG_IMAGES) { a.dbg[b * 16 + 8] = K; a.dbg[b * 16 + 9] = M; }
    if (tid == 0) {   // the last CTA to leave re-arms the ticket for the next launch on this ctx
        __threadfence();
        if (atomicAdd(a.ticket + 1, 1) == (int)gridDim.x - 1) {
            a.ticket[0] = 0;
            a.ticket[1] = 0;
#pragma unroll
            for (int k = 0; k < 8; ++k) a.status_next[k] = 0;
            __threadfence();
        }
    }
}

// Two builds of the same body.  "latency": up to 64 registers, the whole register file of the SM for the one resident CTA —
// the fastest single launch.  "shared": capped at 32 registers (spills go to L1) so the image's CTA leaves half of the SM's
// registers, threads and shared memory to the bandwidth-bound kernels of another in-flight batch (preprocess / warp CTAs
// co-reside): measured -4 % on a strictly serial stream, +13 % with two batches in flight (fd_ctx_set_sharing).
__global__ void __launch_bounds__(FT, 1) detect_fused_kernel(const __grid_constant__ FusedArgs a) { detect_fused_body(a); }
__global__ void __maxnreg__(32) detect_fused_shared_kernel(const __grid_constant__ FusedArgs a) { detect_fused_body(a); }

// Returns FD_OK and sets *launched; *launched == false means the geometry is not eligible and the caller runs the
// three-kernel path.  est_cap: capacity (faces) of ctx->align_M / ctx->align_ok.
int detect_fused_launch(fd_ctx *ctx, const float *const *heads_dev, int B, float conf_thr, float iou_thr, int est_cap, bool *launched) {
    *launched = false;
    static const bool disabled = getenv("FD_NO_FUSED") != nullptr && getenv("FD_NO_FUSED")[0] == '1';
    if (disabled) return FD_OK;
    const DecodeCfg &d = ctx->dcfg;
    for (int st = 0; st < d.n_strides; ++st)   // 128-bit score loads: H*W % 4 == 0 for every stride, 16-byte aligned score tensors
        if ((d.fh[st] * d.fw[st]) % 4 != 0 || reinterpret_cast<uintptr_t>(heads_dev[3 * st]) % 16 != 0) return FD_OK;
    // images with 1024 < K <= 4096 candidates stay on the device once the ctx has met one (fd_detect_fetch saw a deferred
    // image): from then on the launch reserves the general path's shared memory as well
    static const char *force = getenv("FD_FUSED_GENERAL");
    const bool general_ok = (force ? force[0] == '1' : ctx->crowded) &&
                            FUSED_CTRL_BYTES + sizeof(SmallSmem) <= (size_t)ctx->max_smem_optin;
    const size_t smem = FUSED_CTRL_BYTES + (general_ok ? std::max(sizeof(FusedSmem), sizeof(SmallSmem)) : sizeof(FusedSmem));
    if (smem > (size_t)ctx->max_smem_optin) return FD_OK;
    FD_TRY(ticket_buffer(ctx));
    {   // a fresh allocation must not hold a stale tag that could match a future epoch
        const void *before = ctx->scan_agg.p;
        FD_TRY(ctx->scan_agg.reserve(sizeof(u64) * (size_t)B));
        if (ctx->scan_agg.p != before) FD_CUDA(cudaMemsetAsync(ctx->scan_agg.p, 0, ctx->scan_agg.cap, ctx->stream));
    }
    FusedArgs a;
    a.c = d;
    for (int i = 0; i < 3 * FD_MAX_STRIDES; ++i) a.hp.p[i] = i < 3 * d.n_strides ? heads_dev[i] : nullptr;
    a.conf_thr = conf_thr;
    a.iou = make_iou_params(iou_thr, 0);
    a.keys = ctx->cand_keys.as<u64>();
    a.cand_box = ctx->cand_box.as<float4>();
    a.cand_rec = ctx->cand_lmk.as<float>();
    a.counts = ctx->cand_count.as<int>();
    a.keep = ctx->keep_src.as<int>();
    a.keep_count = ctx->keep_count.as<int>();
    a.status = ctx->status();
    a.status_next = reinterpret_cast<int *>(ctx->status_dev.p) + (ctx->status_cur ^ 8);
    a.big_list = ctx->big_list.as<int>();
    a.det_scale = ctx->det_scale_dev.as<float>();
    a.offsets = ctx->out_offsets.as<int>();
    a.out_det = ctx->out_det.as<float>();
    a.out_lmk = ctx->out_lmk.as<float>();
    a.out_frame_idx = ctx->out_frame_idx.as<int>();
    FD_TRY(make_est_const(ctx, &a.ec));
    a.M12 = ctx->align_M.as<double>();
    a.ok = ctx->align_ok.as<uint8_t>();
    a.est_cap = est_cap;
    a.ticket = ctx->tickets.as<int>() + 2;
    a.agg = ctx->scan_agg.as<u64>();
    a.epoch = ++ctx->scan_epoch;
    if (a.epoch == 0) a.epoch = ++ctx->scan_epoch;   // 0 is the "never written" tag
    a.B = B;
    a.general_ok = general_ok ? 1 : 0;
    static const bool dbg_on = getenv("FD_FUSED_DBG") != nullptr;
    static long long *dbg_dev = nullptr;
    a.dbg = nullptr;
    if (dbg_on) {
        if (!dbg_dev) FD_CUDA(cudaMalloc(&dbg_dev, sizeof(long long) * 16 * FUSED_DBG_IMAGES));
        FD_CUDA(cudaMemsetAsync(dbg_dev, 0, sizeof(long long) * 16 * FUSED_DBG_IMAGES, ctx->stream));
        a.dbg = dbg_dev;
    }
    void (*kern)(const FusedArgs) = ctx->share_sms ? detect_fused_shared_kernel : detect_fused_kernel;
    FD_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    FD_TRY(launch_pdl(ctx, kern, dim3(B), dim3(FT), smem, a));
    FD_LAUNCH_CHECK_NAMED(ctx, "detect_fused_kernel");
    if (dbg_on) {
        std::vector<long long> h(16 * (size_t)std::min(B, FUSED_DBG_IMAGES));
        cudaStreamSynchronize(ctx->stream);
        cudaMemcpy(h.data(), dbg_dev, sizeof(long long) * h.size(), cudaMemcpyDeviceToHost);
        long long t0 = h[0];
        for (int b = 0; b < std::min(B, FUSED_DBG_IMAGES); ++b) t0 = std::min(t0, h[16 * b]);
        for (int b = 0; b < std::min(B, FUSED_DBG_IMAGES); ++b) {
            const long long *d = &h[16 * b];
            fprintf(stderr, "[fused dbg] img %3d K=%4lld M=%3lld start+%5.2f scan %5.2f sort %5.2f decode %5.2f nms %6.2f gather %5.2f est %5.2f offs+out %5.2f total %6.2f us\n",
                    b, d[8], d[9], (d[0] - t0) * 1e-3, (d[1] - d[0]) * 1e-3, (d[2] - d[1]) * 1e-3, (d[3] - d[2]) * 1e-3, (d[4] - d[3]) * 1e-3,
                    (d[5] - d[4]) * 1e-3, (d[6] - d[5]) * 1e-3, (d[7] - d[6]) * 1e-3, (d[7] - t0) * 1e-3);
        }
    }
    *launched = true;
    return FD_OK;
}

}  // namespace fd
