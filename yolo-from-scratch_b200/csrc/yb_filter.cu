// yb_filter.cu — K4: fused decode + sigmoid + confidence filter + ordered compaction.
// Reference: the per-scale body of predict(), train.py:1152-1222, and the P3->P4->P5
// concatenation :1227-1229, batched over B images.
//
// Bound: HBM.  Algorithmic bytes (SURVEY 8d): rows*min(row_bytes,32) for the objectness column,
// plus M*row_bytes for the rows that pass and 28*M for the candidate list.
// A tile is 128 consecutive rows of one scale of one image; a CTA owns a GROUP of G consecutive
// tiles (G = 1 for 85-float rows, 8 for 6-float rows: ~24-44 KB of head data per CTA), so that
// every thread has G independent loads in flight.  ONE launch (round 2; round 1 read the objectness column
// twice, in a count kernel and again in an emit kernel):
//   filter_onepass_kernel  objectness test of the group (strided 4-byte loads: every line of a 24-byte-row
//                        head, one 128-byte line per 340-byte row), pass counts per tile, then a DECOUPLED
//                        LOOK-BACK over the groups of the image (order preserving: a group publishes its
//                        count, then its inclusive prefix, in one 64-bit word; successors add up what they
//                        find behind them; group ids are handed out by a per-image ticket so that every
//                        predecessor is already running), in-tile ballot scan, and for the passing rows
//                        decode + class max + box build.  Dense groups are staged in shared memory by ONE
//                        bulk-async copy (cp.async.bulk, mbarrier completion) that is in flight while the
//                        look-back waits: the rows of a group are contiguous in the head tensor, so the
//                        whole group is a single 1-D TMA transfer.  Rows are then read at stride 5+nc words
//                        (odd for nc=80: conflict-free).  The heads cross the HBM interface once.
#include "yb_filter.cuh"

namespace yb {

constexpr int kFTile = 128;    // rows per tile == threads per CTA
constexpr int kFMaxGroup = 8;  // tiles per CTA, at most

__device__ __forceinline__ int group_scale(const FilterArgs& a, uint32_t group) {
    int s = 0;
#pragma unroll
    for (int k = 1; k < YB_MAX_SCALES; ++k)
        if (k < a.S && group >= a.sc[k].group_begin) s = k;
    return s;
}

// first index of the maximum of sigmoid(x[0..nc)) — torch.max(dim=1) semantics (:1189).
// sigmoid is monotone, so the maximum is sigmoid(max logit) and its index is the first maximal
// logit, unless an EARLIER, smaller logit v rounds to the same fp32 probability.  Since
// d/dx ln sigmoid(x) = sigmoid(-x) >= sigmoid(-m) on (-inf, m], two logits whose probabilities
// agree to within k fp32 ulps satisfy m - v <= k * 2^-23 * (1 + e^m); the evaluation error of
// 1/(1+expf(-x)) is below 4 ulp, so k = 16 is safe and only logits above
// lo = m - 2e-6*(1+e^m) are re-evaluated (m <= 14; above that sigmoid saturates and every logit
// above 13 is re-evaluated).  On random heads the re-evaluation practically never runs, which keeps
// the warp converged (the round-1 kernel used a window of 1.0 and spent ~80% of its instructions in
// divergent sigmoid re-evaluations).
// First half: one pass over the logits — maximum m, its first index mi, the runner-up m2 (largest value at any
// other index).  The caller evaluates sigmoid(m) together with the row's other sigmoids and then calls
// class_max_ties, which re-evaluates only when another logit can round to the same probability.
// NaN: torch.max propagates it and returns the index of the first NaN.  A NaN at index 0 stays m (no v > NaN).  Any
// later NaN fails v > m and reaches the runner-up through max.NaN, which keeps it: m2 is NaN after the pass
// exactly when a NaN was seen at an index > 0.  Only then the logits are scanned again for the first NaN; m is
// that NaN (so prob is NaN) and mi its index.  The pass costs what the plain runner-up update cost: one select
// and one max per logit.
__device__ __forceinline__ float fmax_nan(float a, float b) {
    float d;
    asm("max.NaN.f32 %0, %1, %2;" : "=f"(d) : "f"(a), "f"(b));
    return d;
}
template <typename Load>
__device__ __forceinline__ void class_max_logit(int nc, Load ld, float& m, float& m2, int& mi) {
    m = ld(0);
    m2 = -INFINITY;
    mi = 0;
    int c = 1;
    auto step = [&](float v, int idx) {
        const bool gt = v > m;
        m2 = fmax_nan(m2, gt ? m : v);
        if (gt) { m = v; mi = idx; }
    };
    for (; c + 8 <= nc; c += 8) {  // 8 independent loads per step
        float v[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) v[k] = ld(c + k);
#pragma unroll
        for (int k = 0; k < 8; ++k) step(v[k], c + k);
    }
    for (; c < nc; ++c) step(ld(c), c);
    if (m2 != m2) {
        for (c = 0; c + 1 < nc && ld(c) == ld(c); ++c) {}
        m = ld(c);
        mi = c;
    }
}
template <typename Load>
__device__ __forceinline__ void class_max_ties(int nc, Load ld, float m, float m2, int mi, float& prob, int& id) {
    id = mi;   // prob = sigmoid(m) on entry
    if (!(prob > 0.0f)) {
        // NaN: mi is the first NaN.  0: m < -88.73, where expf(-m) overflows; every logit <= m has probability 0
        // as well, so all of them tie and torch.max returns index 0.
        if (prob == 0.0f) id = 0;
        return;
    }
    if (m <= 5.0f && !(m2 > m - 3.1e-4f)) return;  // 2e-6*(1+e^5) < 3.1e-4: the common case without the exponential
    const float lo = (m <= 14.0f) ? m - 2e-6f * (1.0f + expf(m)) : 13.0f;
    if (!(m2 > lo)) return;  // nothing else is close enough to round to the same probability
    for (int c = 0; c < nc; ++c) {  // near-ties on either side of mi (expf need not be monotone to the last ulp)
        const float v = ld(c);
        if (v > lo && c != mi) {
            const float p = sigmoidf_ref(v);
            if (p > prob || (p == prob && c < id)) { prob = p; id = c; }
        }
    }
}

template <typename Load>
__device__ __forceinline__ void class_max(int nc, Load ld, float& prob, int& id) {
    float m, m2;
    int mi;
    class_max_logit(nc, ld, m, m2, mi);
    prob = sigmoidf_ref(m);
    class_max_ties(nc, ld, m, m2, mi, prob, id);
}

// ---- bulk-async (TMA 1-D) staging ------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void bulk_load(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(dst_smem)),
                 "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    uint32_t done;
    do {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done)
            : "r"(smem_u32(bar)), "r"(parity)
            : "memory");
    } while (!done);
}

// ---- decoupled look-back over the groups of one image -------------------------------------------------------
// state word: flag << 32 | value; flag 1 = value is the group's own count, 2 = value is the inclusive prefix.
__device__ __forceinline__ unsigned long long lb_load(const unsigned long long* p) {
    unsigned long long v;
    asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void lb_store(unsigned long long* p, unsigned long long v) {
    asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
// Exclusive prefix of group g (one full warp calls this; st = the image's state row; the group's own count has
// been published already).  Lane l inspects predecessor g-1-l of the current window of 32.
__device__ __forceinline__ int lb_exclusive(const unsigned long long* st, int g, int lane) {
    int prefix = 0;
    for (int hi = g - 1; hi >= 0; hi -= 32) {
        const int k = hi - lane;
        unsigned long long v = 3ull << 32;   // beyond the first group: behaves like an inclusive prefix of 0
        for (;;) {
            if (k >= 0) v = lb_load(st + k);
            const unsigned ready = __ballot_sync(0xffffffffu, (v >> 32) != 0ull);
            const unsigned incl = __ballot_sync(0xffffffffu, (v >> 32) >= 2ull);
            // the nearest predecessor that already knows its inclusive prefix ends the walk; everything nearer
            // must at least have published its count
            const int stop = incl ? __ffs(incl) - 1 : 32;
            const unsigned need = stop >= 32 ? 0xffffffffu : ((2u << stop) - 1u);
            if ((ready & need) == need) {
                int part = (lane <= stop && k >= 0) ? (int)(unsigned)(v & 0xffffffffull) : 0;
                part = __reduce_add_sync(0xffffffffu, part);
                prefix += part;
                if (stop < 32) return prefix;
                break;
            }
        }
    }
    return prefix;
}

// One candidate row -> (box, score, class) at output slot `o` (train.py:1154-1216).  X(c) loads channel c of the row.
template <typename Load>
__device__ __forceinline__ void filter_emit_row(const FilterArgs& a, const FilterScale& L, uint32_t r, size_t o, Load X,
                                                float inv_s, float pt, float pl) {
    uint32_t cell, an, gy, gx;
    L.d_A.divmod(r, cell, an);
    L.d_W.divmod(cell, gy, gx);
    const float aw = __ldg(L.anchors + an * 2), ah = __ldg(L.anchors + an * 2 + 1);
    const float x0 = X(0), x1r = X(1), x2r = X(2), x3r = X(3), x4r = X(4);
    float m, m2;
    int mi;
    class_max_logit(a.nc, [&](int cc) { return X(5 + cc); }, m, m2, mi);
    // the row's six sigmoids 1/(1+expf(-x)) in one basic block: expf is branch-free, the reciprocals are the
    // division's own fast path without its range check (rcp_normal), so the six chains interleave; one check for
    // all of them (x < -87.3: 1+e^-x >= 2^126) redoes the full divisions
    const float d0 = 1.0f + expf(-x0), d1 = 1.0f + expf(-x1r), d2 = 1.0f + expf(-x2r), d3 = 1.0f + expf(-x3r);
    const float d4 = 1.0f + expf(-x4r), d5 = 1.0f + expf(-m);
    float s0 = rcp_normal(d0), s1 = rcp_normal(d1), s2 = rcp_normal(d2), s3 = rcp_normal(d3);
    float s4 = rcp_normal(d4), cprob = rcp_normal(d5);
    if (!(fmaxf(fmaxf(fmaxf(d0, d1), fmaxf(d2, d3)), fmaxf(d4, d5)) < kRcpNormalMax)) {
        s0 = 1.0f / d0; s1 = 1.0f / d1; s2 = 1.0f / d2; s3 = 1.0f / d3; s4 = 1.0f / d4; cprob = 1.0f / d5;
    }
    int cid;
    class_max_ties(a.nc, [&](int cc) { return X(5 + cc); }, m, m2, mi, cprob, cid);
    a.boxes[o] = filter_box(a, L, s0, s1, s2, s3, gx, gy, aw, ah, inv_s, pt, pl);
    a.scores[o] = s4 * cprob;  // :1216
    a.classes[o] = (int64_t)cid;
}

// LONG = false: rows of at most 12 floats; the whole group (8 tiles, <= 48 KB) is staged by one bulk copy issued
//               before anything else — the objectness column touches every sector of such rows anyway — and both
//               phases read shared memory.
// LONG = true:  longer rows (nc = 80: 340 bytes).  Phase A reads the objectness column with strided loads (one
//               128-byte line per row), the group still spans 8 tiles so that only ~25 groups per image take part in
//               the look-back (with one tile per group the look-back's L2 round trips, ~200 participants per image,
//               cost more than the data: 180 us instead of the ~95 us the bytes need).  Phase B first emits the
//               candidates of sparse tiles straight from global memory (no barrier in between: with a barrier per
//               tile the two or three threads that own a candidate stall the whole CTA for ~6 us of dependent
//               loads per tile), then streams the dense tiles (a quarter of the rows or more pass) through ONE
//               shared-memory tile buffer, so that five CTAs per SM keep >200 KB of bulk copies in flight.  When the
//               batch has been dense so far (lb_seen) the first copy starts before phase A.
template <bool LONG, typename T>
__global__ void __launch_bounds__(kFTile) filter_onepass_kernel(const FilterArgs a) {
    extern __shared__ __align__(128) float s_tile[];
    T* s_t = reinterpret_cast<T*>(s_tile);   // staged rows
    __shared__ __align__(8) uint64_t s_bar[2];
    __shared__ int s_wcnt[kFMaxGroup][kFTile / 32];
    __shared__ int s_prefix, s_hint;
    __shared__ unsigned s_gid;
    // row ids (within the group) of the passing rows, in row order, live behind the staged rows
    unsigned short* s_list = reinterpret_cast<unsigned short*>(s_tile + a.sobj_offset);
    const uint32_t b = blockIdx.y;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) {
        mbar_init(&s_bar[0], 1);
        mbar_init(&s_bar[1], 1);
        s_gid = atomicAdd(a.lb_ticket + b, 1u);   // the g-th CTA of the image to start owns group g
        // density hint for long rows: rows and candidates of the groups (of any image) that have finished their
        // objectness pass so far.  A wrong hint only costs bandwidth, never correctness.
        int hint = 0;
        if (LONG && a.stage_ok) {
            const unsigned rows_done = *(volatile unsigned*)(a.lb_seen), cand_done = *(volatile unsigned*)(a.lb_seen + 1);
            hint = rows_done != 0u && (unsigned long long)cand_done * 4ull >= (unsigned long long)rows_done;
        }
        s_hint = hint;
    }
    __syncthreads();
    const uint32_t group = s_gid;
    const int s = group_scale(a, group);
    const FilterScale& L = a.sc[s];
    const uint32_t tile0 = (group - L.group_begin) * a.G;  // within the scale
    const uint32_t ntiles = (L.rows + kFTile - 1) / kFTile;
    const int G = (int)min((uint32_t)a.G, ntiles - tile0);  // tiles of this group
    const uint32_t row0 = tile0 * kFTile;
    const uint32_t nrows = min((uint32_t)(G * kFTile), L.rows - row0);
    const size_t base = ((size_t)b * L.rows + row0) * a.row;  // element offset of the group
    const T* g = reinterpret_cast<const T*>(L.pred) + base;
    unsigned long long* st = a.lb_state + (size_t)b * a.groups_per_img;
    const uint32_t tile_fl = (uint32_t)kFTile * a.row;        // elements of a full tile
    constexpr uint32_t VM = kVec<T> - 1u;                     // 16-byte alignment mask, in elements
    constexpr uint32_t ES = sizeof(T);

    // tile k of the group as a bulk-copy job: rows, floats, source, 16-byte alignment
    auto tile_rows = [&](int k) { return min((uint32_t)kFTile, nrows - (uint32_t)k * kFTile); };
    auto tile_bulk_ok = [&](int k) { return ((base + (size_t)k * tile_fl) & VM) == 0 && ((tile_rows(k) * a.row) & VM) == 0; };
    int pending = -1;               // tile whose bulk copy is in flight / has landed in the buffer (all threads agree)
    uint32_t parity = 0u;

    if (!LONG) {   // the whole group up front
        const uint32_t nfl = nrows * a.row;
        if ((base & VM) == 0 && (nfl & VM) == 0) {
            if (threadIdx.x == 0) bulk_load(s_t, g, nfl * ES, &s_bar[0]);
            mbar_wait(&s_bar[0], 0);
        } else {
            for (uint32_t e = threadIdx.x; e < nfl; e += kFTile) s_t[e] = g[e];
            __syncthreads();
        }
    } else if (s_hint && tile_bulk_ok(0)) {   // speculative: the first tile
        if (threadIdx.x == 0) bulk_load(s_t, g, tile_rows(0) * a.row * ES, &s_bar[0]);
        pending = 0;
    }

    // phase A: objectness test of this thread's row in every tile of the group (the only pass over the column).
    // sigmoid(x) > conf is decided from the logit when x is clearly on one side of logit(conf) (the fp32
    // sigmoid is within a few ulp of the real one, so a margin of obj_margin in x cannot flip the comparison);
    // rows inside the margin evaluate the reference expression.  The lower test is inclusive: without a margin
    // (obj_lo = -inf) a row with x = -inf still evaluates sigmoid(-inf) = 0 > conf, which holds for conf < 0.
    float xo[kFMaxGroup];
#pragma unroll
    for (int k = 0; k < kFMaxGroup; ++k) {
        const uint32_t rl = k * kFTile + threadIdx.x;
        xo[k] = __int_as_float(0x7fc00000);   // NaN: fails both quick tests and the exact one
        if (k < G && rl < nrows) xo[k] = LONG ? ldg_f(g + (size_t)rl * a.row + 4) : to_f32(s_t[rl * a.row + 4]);
    }
    unsigned mybal[kFMaxGroup];
#pragma unroll
    for (int k = 0; k < kFMaxGroup; ++k) {
        mybal[k] = 0u;
        if (k < G) {
            bool pass = xo[k] > a.obj_hi;
            if (!pass && xo[k] >= a.obj_lo) pass = sigmoidf_ref(xo[k]) > a.conf;   // :1157,:1166-1167 objectness only
            const unsigned bal = __ballot_sync(0xffffffffu, pass);
            mybal[k] = bal;
            if (lane == 0) s_wcnt[k][warp] = __popc(bal);
        }
    }
    __syncthreads();
    // offsets of this warp's rows of tile k in the group's list, per-tile counts, the group's total
    int woff[kFMaxGroup], tcnt[kFMaxGroup];
    int total = 0;
#pragma unroll
    for (int k = 0; k < kFMaxGroup; ++k) {
        woff[k] = total;
        tcnt[k] = 0;
        if (k < G) {
#pragma unroll
            for (int w = 0; w < kFTile / 32; ++w) {
                const int c = s_wcnt[k][w];
                if (w < warp) woff[k] += c;
                tcnt[k] += c;
            }
            total += tcnt[k];
        }
    }
    // publish the group's count (the first group's count is its inclusive prefix)
    if (threadIdx.x == 0) {
        lb_store(st + group, ((group == 0 ? 2ull : 1ull) << 32) | (unsigned)total);
        if (LONG) { atomicAdd(a.lb_seen, nrows); atomicAdd(a.lb_seen + 1, (unsigned)total); }
    }
    // LONG: a tile is staged when at least a quarter of its rows pass; start the first one unless a copy is in flight
    unsigned dense_mask = 0u;
#pragma unroll
    for (int k = 0; k < kFMaxGroup; ++k)
        if (LONG && k < G && a.stage_ok && tcnt[k] > 0 && tcnt[k] * 4 >= (int)tile_rows(k) && tile_bulk_ok(k)) dense_mask |= 1u << k;
    if (LONG && pending < 0 && dense_mask) {
        const int k = __ffs(dense_mask) - 1;
        if (threadIdx.x == 0) bulk_load(s_t, g + (size_t)k * tile_fl, tile_rows(k) * a.row * ES, &s_bar[0]);
        pending = k;
    }
#pragma unroll
    for (int k = 0; k < kFMaxGroup; ++k)
        if (k < G && ((mybal[k] >> lane) & 1u))
            s_list[woff[k] + __popc(mybal[k] & ((1u << lane) - 1u))] = (unsigned short)(k * kFTile + threadIdx.x);
    if (warp == 0) {
        const int p = group == 0 ? 0 : lb_exclusive(st, (int)group, lane);
        if (lane == 0) {
            s_prefix = p;
            if (group != 0) lb_store(st + group, (2ull << 32) | (unsigned)(p + total));
            if (group + 1 == a.groups_per_img) {
                const int tot = p + total;
                a.counts[b] = tot < a.cap ? tot : a.cap;
            }
        }
    }
    __syncthreads();
    const int prefix = s_prefix;

    // phase B: emit, one passing row per thread and step (the list is dense: no idle lanes at any pass rate)
    float inv_s = 1.0f, pt = 0.0f, pl = 0.0f;
    if (a.letterbox) {
        inv_s = 1.0f / a.letterbox[b * 3 + 0];
        pt = a.letterbox[b * 3 + 1];
        pl = a.letterbox[b * 3 + 2];
    }
    const int n_emit = min(total, a.cap - prefix);
    if (!LONG) {
#pragma unroll 1
        for (int c = threadIdx.x; c < n_emit; c += kFTile) {
            const uint32_t rl = s_list[c];
            const T* x = s_t + rl * a.row;
            filter_emit_row(a, L, row0 + rl, (size_t)b * a.cap + prefix + c, [&](int ch) { return to_f32(x[ch]); }, inv_s, pt, pl);
        }
        return;
    }
    // sparse tiles: straight from global memory, every candidate of the group at once, no barrier
    if (pending >= 0 && !((dense_mask >> pending) & 1u) && tcnt[pending] > 0) dense_mask |= 1u << pending;   // a speculative copy that is useful after all
#pragma unroll 1
    for (int c = threadIdx.x; c < n_emit; c += kFTile) {
        const uint32_t rl = s_list[c];
        if ((dense_mask >> (rl / kFTile)) & 1u) continue;
        const T* x = g + (size_t)rl * a.row;
        filter_emit_row(a, L, row0 + rl, (size_t)b * a.cap + prefix + c, [&](int ch) { return ldg_f(x + ch); }, inv_s, pt, pl);
    }
    // dense tiles: one bulk copy at a time through the tile buffer
    int off = 0;   // list offset of tile k
#pragma unroll 1
    for (int k = 0; k < G; ++k) {
        const int n_k = max(0, min(tcnt[k], n_emit - off));
        if ((dense_mask >> k) & 1u) {
            if (pending >= 0 && pending != k) {   // a speculative copy of an empty tile: it must land before the next one
                mbar_wait(&s_bar[0], parity);
                parity ^= 1u;
                pending = -1;
            }
            if (pending != k) {
                if (threadIdx.x == 0) bulk_load(s_t, g + (size_t)k * tile_fl, tile_rows(k) * a.row * ES, &s_bar[0]);
            }
            mbar_wait(&s_bar[0], parity);
            parity ^= 1u;
            pending = -1;
            const T* xb = s_t - (size_t)k * tile_fl;
#pragma unroll 1
            for (int c = threadIdx.x; c < n_k; c += kFTile) {
                const uint32_t rl = s_list[off + c];
                const T* x = xb + (size_t)rl * a.row;
                filter_emit_row(a, L, row0 + rl, (size_t)b * a.cap + prefix + off + c, [&](int ch) { return to_f32(x[ch]); }, inv_s, pt, pl);
            }
            __syncthreads();   // the buffer is free again
            const unsigned rest = dense_mask >> (k + 1);
            if (rest) {          // next dense tile: start its copy right away
                const int k2 = k + __ffs(rest);
                if (threadIdx.x == 0) bulk_load(s_t, g + (size_t)k2 * tile_fl, tile_rows(k2) * a.row * ES, &s_bar[0]);
                pending = k2;
            }
        }
        off += tcnt[k];
    }
    if (pending >= 0) mbar_wait(&s_bar[0], parity);   // a speculative copy nobody needed must still land before the CTA exits
}

// ------------------------------------------------------------------------------------------------
// NCHW heads (f-2): (B, A*row, H, W), the head conv's own output.  A tile is 128 consecutive CELLS of
// one scale with all A anchors (128*A canonical rows): thread <-> cell, so every load of a channel
// plane is a fully coalesced 128-byte line per warp and no shared-memory staging is needed.  The
// candidate order stays the canonical (cell, anchor) order of the reference layout.
// ------------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(kFTile) filter_count_nchw_kernel(const FilterArgs a, const FilterNchw n) {
    __shared__ int s_red[kFTile / 32];
    const uint32_t tile = blockIdx.x, b = blockIdx.y;
    const int s = nchw_tile_scale(a, n, tile);
    const FilterScale& L = a.sc[s];
    const uint32_t cell = (tile - n.tile_begin[s]) * kFTile + threadIdx.x;
    int cnt = 0;
    if (cell < L.hw) {
        float x[YB_MAX_ANCHORS];
#pragma unroll
        for (int an = 0; an < YB_MAX_ANCHORS; ++an)
            if (an < a.A) x[an] = ldg_f(reinterpret_cast<const T*>(L.pred) + ((size_t)(b * (uint32_t)a.A + an) * a.row + 4) * L.hw + cell);
#pragma unroll
        for (int an = 0; an < YB_MAX_ANCHORS; ++an)
            if (an < a.A) cnt += sigmoidf_ref(x[an]) > a.conf ? 1 : 0;  // :1157,:1166-1167 objectness only
    }
    cnt = __reduce_add_sync(0xffffffffu, cnt);
    if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = cnt;
    __syncthreads();
    if (threadIdx.x == 0) {
        int tot = 0;
#pragma unroll
        for (int k = 0; k < kFTile / 32; ++k) tot += s_red[k];
        a.tile_counts[b * n.tiles_per_img + tile] = tot;
    }
}

template <typename T>
__global__ void __launch_bounds__(kFTile) filter_emit_nchw_kernel(const FilterArgs a, const FilterNchw n) {
    __shared__ int s_red[kFTile / 32];
    __shared__ int s_wsum[kFTile / 32];
    const uint32_t tile = blockIdx.x, b = blockIdx.y;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int* tc = a.tile_counts + b * n.tiles_per_img;
    int part = 0;
    for (uint32_t t = threadIdx.x; t < tile; t += kFTile) part += tc[t];
    part = __reduce_add_sync(0xffffffffu, part);
    if (lane == 0) s_red[warp] = part;
    __syncthreads();
    int prefix = 0;
#pragma unroll
    for (int k = 0; k < kFTile / 32; ++k) prefix += s_red[k];
    const int count = tc[tile];
    if (tile == n.tiles_per_img - 1 && threadIdx.x == 0) {
        const int tot = prefix + count;
        a.counts[b] = tot < a.cap ? tot : a.cap;
    }
    if (count == 0) return;

    const int s = nchw_tile_scale(a, n, tile);
    const FilterScale& L = a.sc[s];
    const uint32_t cell = (tile - n.tile_begin[s]) * kFTile + threadIdx.x;
    const bool valid = cell < L.hw;
    const T* plane0 = reinterpret_cast<const T*>(L.pred) + (size_t)b * a.A * a.row * L.hw + (valid ? cell : 0u);  // channel 0, anchor 0
    const size_t hw = L.hw;

    // phase A: objectness of this cell for every anchor
    float so[YB_MAX_ANCHORS];
    unsigned passmask = 0u;
#pragma unroll
    for (int an = 0; an < YB_MAX_ANCHORS; ++an) {
        so[an] = 0.0f;
        if (an < a.A && valid) so[an] = ldg_f(plane0 + ((size_t)an * a.row + 4) * hw);
    }
#pragma unroll
    for (int an = 0; an < YB_MAX_ANCHORS; ++an) {
        if (an < a.A && valid) {
            so[an] = sigmoidf_ref(so[an]);
            if (so[an] > a.conf) passmask |= 1u << an;
        }
    }
    // exclusive scan of the per-cell pass counts: canonical order is (cell, anchor)
    const int mine = __popc(passmask);
    int inc = mine;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int v = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += v;
    }
    if (lane == 31) s_wsum[warp] = inc;
    __syncthreads();
    int pos = prefix + inc - mine;
    for (int k = 0; k < warp; ++k) pos += s_wsum[k];
    if (!passmask) return;

    float inv_s = 1.0f, pt = 0.0f, pl = 0.0f;
    if (a.letterbox) {
        inv_s = 1.0f / a.letterbox[b * 3 + 0];
        pt = a.letterbox[b * 3 + 1];
        pl = a.letterbox[b * 3 + 2];
    }
    uint32_t gy, gx;
    L.d_W.divmod(cell, gy, gx);
#pragma unroll
    for (int an = 0; an < YB_MAX_ANCHORS; ++an) {
        if (an >= a.A || !((passmask >> an) & 1u)) continue;
        if (pos >= a.cap) break;
        const T* x = plane0 + (size_t)an * a.row * hw;
        const float aw = __ldg(L.anchors + an * 2), ah = __ldg(L.anchors + an * 2 + 1);
        const float x0 = ldg_f(x), x1r = ldg_f(x + hw), x2r = ldg_f(x + 2 * hw), x3r = ldg_f(x + 3 * hw);
        float cprob;
        int cid;
        class_max(a.nc, [&](int c) { return ldg_f(x + (size_t)(5 + c) * hw); }, cprob, cid);
        const float bx = decode_xy(x0, (float)gx, L.inv_w);
        const float by = decode_xy(x1r, (float)gy, L.inv_h);
        const float bw = decode_wh(x2r, aw, a.inv_img);
        const float bh = decode_wh(x3r, ah, a.inv_img);
        const float xc = bx * a.img, yc = by * a.img, wp = bw * a.img, hp = bh * a.img;
        float x1 = xc - wp * 0.5f, y1 = yc - hp * 0.5f, x2 = xc + wp * 0.5f, y2 = yc + hp * 0.5f;
        if (a.letterbox) {
            x1 = (x1 - pl) * inv_s; y1 = (y1 - pt) * inv_s;
            x2 = (x2 - pl) * inv_s; y2 = (y2 - pt) * inv_s;
        }
        const size_t o = (size_t)b * a.cap + pos;
        a.boxes[o] = make_float4(x1, y1, x2, y2);
        a.scores[o] = so[an] * cprob;
        a.classes[o] = (int64_t)cid;
        ++pos;
    }
}

static int filter_fill(const yb_heads_desc* d, FilterArgs& a) {
    // tiles per CTA: kFMaxGroup in the reference layout (short rows stage the whole group, long rows stream tile by
    // tile); NCHW keeps its own cell tiling
    return yb::filter_fill(d, a, kFMaxGroup, kFTile);   // (4 or 2 tiles per group measured no faster: 28 / 28 / 38 us on configs[1])
}

}  // namespace yb

namespace yb {
template <typename T>
static int filter_launch(const yb_heads_desc* d, FilterArgs& a, void* ws, cudaStream_t st) {
    // staging sizes follow the element size: half rows take half the bytes, so rows of up to 24 halves stage the
    // whole group and a long-row tile buffer takes half the shared memory (more CTAs per SM)
    const size_t es = sizeof(T);
    const size_t tile_fl = ((size_t)kFTile * a.row + 31) / 32 * 32;   // elements
    const bool long_rows = (size_t)a.G * kFTile * a.row * es > 48 * 1024;
    size_t smem = long_rows ? tile_fl * es : (size_t)a.G * kFTile * a.row * es;
    a.stage_ok = smem <= 200 * 1024;   // else: rows so long that one tile does not fit; the emit reads global memory
    if (!a.stage_ok) smem = 0;
    smem = (smem + 127) / 128 * 128;
    a.sobj_offset = (uint32_t)(smem / sizeof(float));
    smem += (size_t)a.G * kFTile * sizeof(float);   // NCHW: sigmoid(obj) scratch; reference layout: u16 row list (half of it)
    if (a.nchw) {
        const FilterNchw n = filter_cell_tiles(a, d->S, kFTile);   // <= tiles_per_img of the row tiling: the workspace is large enough
        dim3 ngrid(n.tiles_per_img, d->B);
        YB_LAUNCH("filter_count_nchw_kernel", st, filter_count_nchw_kernel<T><<<ngrid, kFTile, 0, st>>>(a, n));
        YB_LAUNCH("filter_emit_nchw_kernel", st, filter_emit_nchw_kernel<T><<<ngrid, kFTile, 0, st>>>(a, n));
        return 0;
    }
    dim3 grid(a.groups_per_img, d->B);
    a.lb_state = reinterpret_cast<unsigned long long*>(ws);
    a.lb_ticket = reinterpret_cast<unsigned int*>(a.lb_state + (size_t)d->B * a.groups_per_img);
    a.lb_seen = a.lb_ticket + d->B;
    YB_CUDA(cudaMemsetAsync(ws, 0, (size_t)d->B * a.groups_per_img * sizeof(unsigned long long) + ((size_t)d->B + 2) * sizeof(unsigned int), st));
    const size_t dyn = smem;
    if (long_rows) {
        if (dyn > 48 * 1024)
            YB_CUDA(cudaFuncSetAttribute(filter_onepass_kernel<true, T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn));
        YB_LAUNCH("filter_onepass_kernel", st, (filter_onepass_kernel<true, T><<<grid, kFTile, dyn, st>>>(a)));
    } else {
        if (dyn > 48 * 1024)
            YB_CUDA(cudaFuncSetAttribute(filter_onepass_kernel<false, T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn));
        YB_LAUNCH("filter_onepass_kernel", st, (filter_onepass_kernel<false, T><<<grid, kFTile, dyn, st>>>(a)));
    }
    return 0;
}
}  // namespace yb

extern "C" size_t yb_filter_workspace_bytes(const yb_heads_desc* d) {
    yb::FilterArgs a;
    if (yb::filter_fill(d, a)) return 0;
    // NCHW: per-tile counts (4 B); reference layout: look-back state (8 B per group) + one ticket per image
    const size_t nchw = (size_t)d->B * a.tiles_per_img * sizeof(int);
    const size_t lb = (size_t)d->B * a.groups_per_img * sizeof(unsigned long long) + ((size_t)d->B + 2) * sizeof(unsigned int);
    return (nchw > lb ? nchw : lb) + 16;
}

extern "C" int yb_filter_compact(const yb_heads_desc* d, float conf_thres, const float* letterbox,
                                 float* boxes, float* scores, int64_t* classes, int* counts, int cap,
                                 void* ws, size_t ws_bytes, void* stream) {
    using namespace yb;
    FilterArgs a;
    int rc = filter_fill(d, a);
    if (rc) return rc;
    if (d->B == 0) return 0;
    YB_CHECK_ARG(boxes && scores && classes && counts && ws && cap > 0, "filter: null output");
    YB_CHECK_ARG(aligned16(boxes) && (reinterpret_cast<uintptr_t>(ws) & 7u) == 0, "filter: boxes must be 16-byte, the workspace 8-byte aligned");
    for (int s = 0; s < d->S; ++s)
        YB_CHECK_ARG(d->pred[s] && d->anchors[s] && aligned16(d->pred[s]), "filter: bad tensor at scale %d", s);
    if (ws_bytes < yb_filter_workspace_bytes(d)) {
        set_error("filter: workspace too small");
        return YB_EWORKSPACE;
    }
    YB_CHECK_ARG(d->B <= 65535, "filter: B too large");
    a.cap = cap; a.conf = conf_thres; a.letterbox = letterbox;
    {
        // sigmoid(x) > conf  <=>  x > logit(conf) in real arithmetic; 1/(1+expf(-x)) is within 4 ulp of it, i.e.
        // within 2^-21 relative, which moves the crossing point by at most 2^-21/(1-s) (s > 1/2) or 2^-21/s in x.
        // A margin 64x that wide is used; thresholds too close to 0 or 1 always take the exact expression.
        const double c = (double)conf_thres;
        a.obj_lo = -INFINITY; a.obj_hi = INFINITY;
        if (c > 1e-4 && c < 1.0 - 1e-4) {
            const double lg = log(c / (1.0 - c));
            const double m = 64.0 * 4.8e-7 / (c < 0.5 ? c : 1.0 - c) + 1e-5 * fabs(lg) + 1e-6;
            a.obj_lo = (float)(lg - m); a.obj_hi = (float)(lg + m);
        }
    }
    a.tile_counts = reinterpret_cast<int*>(ws);
    a.boxes = reinterpret_cast<float4*>(boxes); a.scores = scores; a.classes = classes; a.counts = counts;
    cudaStream_t st = (cudaStream_t)stream;
    YB_DISPATCH_DTYPE(d->dtype, T, return filter_launch<T>(d, a, ws, st));
    return 0;
}
