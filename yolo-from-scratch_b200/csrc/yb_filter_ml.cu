// yb_filter_ml.cu — multi-label candidate filter with a per-image top-K cap (include/yolo_b200.h, yb_filter_multilabel,
// states the semantics).  A candidate is a (row, class) pair whose score fp32(sigmoid(obj) * sigmoid(cls_c)) passes
// conf; an image keeps at most K of them, the best by (score descending, candidate order), emitted in candidate order.
//
// No candidate list is ever stored: the workspace grows with the rows, not with rows * nc.  Scores are >= 0 and
// <= 1, so their bit patterns are ordered like their values and fit 30 bits: three 10-bit radix digits.  Every kernel
// runs over cell tiles (thread <-> cell, all A anchors, the NCHW kernels' tiling of yb_filter.cu) and recomputes the
// scores of its candidates from the heads:
//   filter_ml_count_kernel   candidates per thread and per tile, histogram of digit 1 per image (shared memory,
//                            flushed with atomics)
//   filter_ml_select_kernel  one CTA per image: N_b <= K -> "keep all"; otherwise the bin of digit L that holds the
//                            K-th largest key (a suffix scan over the 1024 bins); level 3 yields the K-th key t itself
//   filter_ml_refine_kernel  capped images only: level 2 / 3 histogram the next digit of the keys inside the bin found
//                            so far; level 4 counts per thread and tile the keys above t and equal to t
//   filter_ml_emit_kernel    exclusive prefix over the tiles of kept candidates (keys above t, plus ties taken in
//                            candidate order), then every thread writes its kept candidates in candidate order
// Refinement launches run unconditionally (images under the cap return at once), so the call never synchronises and
// is capturable; they are skipped only when K >= rows * nc, where no image can exceed the cap.
#include "yb_filter.cuh"

namespace yb {

constexpr int kMlTile = 128;       // cells per tile == threads per CTA
constexpr int kMlBins = 1024;      // one 10-bit digit of a 30-bit score key
constexpr int kMlSelect = 1024;    // threads of the select kernel: one per bin

enum { ML_MODE, ML_PREFIX, ML_NEED, ML_ABOVE, ML_T, ML_TIES, ML_WORDS = 8 };   // per-image state words

struct MlArgs {
    FilterNchw n;        // cell tiles of every scale
    int K;
    unsigned* hist;      // (B, 3, kMlBins): digit histograms of levels 1..3
    int* state;          // (B, ML_WORDS): mode (1 = capped), digits found so far, keys still needed in the current bin,
                         //   keys above it, the K-th key t, ties at t to keep
    int* tile_above;     // (B, tiles): candidates per tile (keep all) or keys > t (capped)
    int* tile_ties;      // (B, tiles): 0 or keys == t
    int* thr_above;      // (B, tiles * kMlTile): the same per thread
    int* thr_ties;
    int* totals;         // (B) or null
};

// Offset of channel 0 of row r of image b and the distance between its channels.  head_row_offset addresses the same
// element, but its NCHW split also lets r run past image b; in these kernels that costs the multi-label filter 1-2%
// (tools/bench_multilabel.py, nc = 80, B = 64, 640^2 on a B200 at a 1000 W power limit: 1.278 -> 1.302 ms).
__device__ __forceinline__ size_t ml_row(const FilterArgs& a, const FilterScale& L, uint32_t b, uint32_t r, uint32_t& cstride) {
    if (!a.nchw) {
        cstride = 1u;
        return ((size_t)b * L.img_rows + r) * a.row;
    }
    uint32_t cell, an;
    L.d_A.divmod(r, cell, an);
    cstride = L.HW;
    return ((size_t)(b * (uint32_t)a.A + an) * a.row) * L.HW + cell;
}

// Calls f(an, c, key) for every candidate of cell `cell` (scale L, image b) in candidate order, anchors then classes
// ascending; key = the bits of score = fp32(sigmoid(obj) * sigmoid(cls_c)) > conf.  The objectness test is the
// single-label filter's sigmoid(obj) > conf; a NaN logit fails every test.
template <typename T, typename F>
__device__ __forceinline__ void ml_cell(const FilterArgs& a, const FilterScale& L, uint32_t b, uint32_t cell, F f) {
    for (int an = 0; an < a.A; ++an) {
        uint32_t cs;
        const T* x = reinterpret_cast<const T*>(L.pred) + ml_row(a, L, b, cell * (uint32_t)a.A + an, cs);
        const float so = sigmoidf_ref(ldg_f(x + (size_t)4 * cs));
        if (!(so > a.conf)) continue;
        const T* xc = x + (size_t)5 * cs;
        int c = 0;
        for (; c + 8 <= a.nc; c += 8) {   // 8 independent loads and sigmoid chains per step
            float v[8], s[8];
#pragma unroll
            for (int k = 0; k < 8; ++k) v[k] = ldg_f(xc + (size_t)(c + k) * cs);
            sigmoid_ref_batch<8>(v, s);
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                const float sc = so * s[k];
                if (sc > a.conf) f(an, c + k, __float_as_uint(sc));
            }
        }
        for (; c < a.nc; ++c) {
            const float sc = so * sigmoidf_ref(ldg_f(xc + (size_t)c * cs));
            if (sc > a.conf) f(an, c, __float_as_uint(sc));
        }
    }
}

// The scale of cell tile `tile` (nchw_tile_scale's choice) and this thread's cell in it.  Selected through static
// indices only: a dynamic index into a kernel parameter array copies the array to local memory.
__device__ __forceinline__ FilterScale ml_tile(const FilterArgs& a, const FilterNchw& n, uint32_t tile, uint32_t& cell) {
    FilterScale L = a.sc[0];
    uint32_t t0 = 0;
#pragma unroll
    for (int k = 1; k < YB_MAX_SCALES; ++k)
        if (k < a.S && tile >= n.tile_begin[k]) {
            L = a.sc[k];
            t0 = n.tile_begin[k];
        }
    cell = (tile - t0) * kMlTile + threadIdx.x;
    return L;
}

// Exclusive scan of v over the NT threads of the block; total receives the sum.  Every thread must call it.
template <int NT>
__device__ __forceinline__ int ml_block_scan(int v, int* s_w, int& total) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int u = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += u;
    }
    if (lane == 31) s_w[warp] = inc;
    __syncthreads();
    int before = 0;
    total = 0;
#pragma unroll
    for (int k = 0; k < NT / 32; ++k) {
        const int w = s_w[k];
        if (k < warp) before += w;
        total += w;
    }
    __syncthreads();   // s_w may be reused
    return before + inc - v;
}

__device__ __forceinline__ void ml_flush_hist(const unsigned* s_hist, unsigned* gh) {
    for (int i = threadIdx.x; i < kMlBins; i += kMlTile)
        if (s_hist[i]) atomicAdd(gh + i, s_hist[i]);
}

template <typename T>
__global__ void __launch_bounds__(kMlTile) filter_ml_count_kernel(const FilterArgs a, const MlArgs m) {
    __shared__ unsigned s_hist[kMlBins];
    __shared__ int s_w[kMlTile / 32];
    const uint32_t tile = blockIdx.x, b = blockIdx.y;
    for (int i = threadIdx.x; i < kMlBins; i += kMlTile) s_hist[i] = 0u;
    __syncthreads();
    uint32_t cell;
    const FilterScale L = ml_tile(a, m.n, tile, cell);
    int cnt = 0;
    if (cell < L.HW)
        ml_cell<T>(a, L, b, cell, [&](int, int, uint32_t key) {
            ++cnt;
            atomicAdd(&s_hist[key >> 20], 1u);
        });
    const size_t ti = (size_t)b * m.n.tiles_per_img + tile;
    m.thr_above[ti * kMlTile + threadIdx.x] = cnt;
    m.thr_ties[ti * kMlTile + threadIdx.x] = 0;
    int tot;
    ml_block_scan<kMlTile>(cnt, s_w, tot);   // its barriers also complete the histogram
    if (threadIdx.x == 0) {
        m.tile_above[ti] = tot;
        m.tile_ties[ti] = 0;
    }
    ml_flush_hist(s_hist, m.hist + (size_t)b * 3 * kMlBins);
}

// Level L of the radix select for image blockIdx.x.  Thread j holds bin 1023 - j, so an inclusive scan over j counts
// the keys in bins >= that bin; the one bin with above < need <= above + count holds the K-th key.
__global__ void __launch_bounds__(kMlSelect) filter_ml_select_kernel(const MlArgs m, int level, int* counts) {
    __shared__ int s_w[kMlSelect / 32];
    const uint32_t b = blockIdx.x;
    int* st = m.state + (size_t)b * ML_WORDS;
    if (level > 1 && st[ML_MODE] == 0) return;   // keep all
    int need = level == 1 ? m.K : st[ML_NEED];   // read before any thread writes the state
    const int i = kMlBins - 1 - (int)threadIdx.x;
    const int v = (int)m.hist[((size_t)b * 3 + level - 1) * kMlBins + i];
    int total;
    const int above = ml_block_scan<kMlSelect>(v, s_w, total);   // keys in bins > i
    if (level == 1) {
        if (threadIdx.x == 0) {
            counts[b] = total < m.K ? total : m.K;
            if (m.totals) m.totals[b] = total;
            st[ML_MODE] = total > m.K ? 1 : 0;
            st[ML_ABOVE] = 0;
            st[ML_PREFIX] = 0;
        }
        if (total <= m.K) return;
    }
    __syncthreads();
    if (above < need && need <= above + v) {
        need -= above;
        const int prefix = (level == 1 ? 0 : st[ML_PREFIX] << 10) | i;
        st[ML_ABOVE] += above;
        st[ML_NEED] = need;
        st[ML_PREFIX] = prefix;
        if (level == 3) {
            st[ML_T] = prefix;
            st[ML_TIES] = need;   // ties at t to keep: 1 <= need <= v
        }
    }
}

// level 2 / 3: histogram of digit `level` over the keys of the bin found so far; level 4: keys > t and == t per thread
// and per tile
template <typename T>
__global__ void __launch_bounds__(kMlTile) filter_ml_refine_kernel(const FilterArgs a, const MlArgs m, int level) {
    __shared__ unsigned s_hist[kMlBins];
    __shared__ int s_w[kMlTile / 32];
    const uint32_t tile = blockIdx.x, b = blockIdx.y;
    const int* st = m.state + (size_t)b * ML_WORDS;
    if (st[ML_MODE] == 0) return;   // keep all: the count kernel's numbers stand
    uint32_t cell;
    const FilterScale L = ml_tile(a, m.n, tile, cell);
    if (level < 4) {
        for (int i = threadIdx.x; i < kMlBins; i += kMlTile) s_hist[i] = 0u;
        __syncthreads();
        const uint32_t prefix = (uint32_t)st[ML_PREFIX];
        const int shift = level == 2 ? 20 : 10;   // keys of the bin: key >> shift == prefix; digit: the next 10 bits
        if (cell < L.HW)
            ml_cell<T>(a, L, b, cell, [&](int, int, uint32_t key) {
                if ((key >> shift) == prefix) atomicAdd(&s_hist[(key >> (shift - 10)) & (kMlBins - 1)], 1u);
            });
        __syncthreads();
        ml_flush_hist(s_hist, m.hist + ((size_t)b * 3 + level - 1) * kMlBins);
        return;
    }
    const uint32_t t = (uint32_t)st[ML_T];
    int above = 0, ties = 0;
    if (cell < L.HW)
        ml_cell<T>(a, L, b, cell, [&](int, int, uint32_t key) {
            above += key > t ? 1 : 0;
            ties += key == t ? 1 : 0;
        });
    const size_t ti = (size_t)b * m.n.tiles_per_img + tile;
    m.thr_above[ti * kMlTile + threadIdx.x] = above;
    m.thr_ties[ti * kMlTile + threadIdx.x] = ties;
    int ta, tt;
    ml_block_scan<kMlTile>(above, s_w, ta);
    ml_block_scan<kMlTile>(ties, s_w, tt);
    if (threadIdx.x == 0) {
        m.tile_above[ti] = ta;
        m.tile_ties[ti] = tt;
    }
}

template <typename T>
__global__ void __launch_bounds__(kMlTile) filter_ml_emit_kernel(const FilterArgs a, const MlArgs m) {
    __shared__ int s_w[kMlTile / 32];
    const uint32_t tile = blockIdx.x, b = blockIdx.y;
    const int* st = m.state + (size_t)b * ML_WORDS;
    const bool capped = st[ML_MODE] != 0;
    const int ties_needed = capped ? st[ML_TIES] : 0;
    const uint32_t t = capped ? (uint32_t)st[ML_T] : 0u;
    const size_t tb = (size_t)b * m.n.tiles_per_img;
    // kept candidates of the tiles before this one: their keys above t plus the ties they keep, ties being kept in
    // candidate order until ties_needed are taken
    int kept_before = 0, ties_before = 0;
    for (uint32_t k0 = 0; k0 < tile; k0 += kMlTile) {
        const uint32_t k = k0 + threadIdx.x;
        const int ab = k < tile ? m.tile_above[tb + k] : 0, ti = k < tile ? m.tile_ties[tb + k] : 0;
        int tsum, ksum;
        const int tbase = ties_before + ml_block_scan<kMlTile>(ti, s_w, tsum);
        ml_block_scan<kMlTile>(ab + min(max(ties_needed - tbase, 0), ti), s_w, ksum);
        kept_before += ksum;
        ties_before += tsum;
    }
    const size_t th = (tb + tile) * kMlTile + threadIdx.x;
    const int my_above = m.thr_above[th], my_ties = m.thr_ties[th];
    int tot;
    const int tie_base = ties_before + ml_block_scan<kMlTile>(my_ties, s_w, tot);
    const int my_tk = min(max(ties_needed - tie_base, 0), my_ties);   // ties this thread keeps: its first my_tk
    int pos = kept_before + ml_block_scan<kMlTile>(my_above + my_tk, s_w, tot);
    if (my_above + my_tk == 0) return;

    uint32_t cell;
    const FilterScale L = ml_tile(a, m.n, tile, cell);
    float inv_s = 1.0f, pt = 0.0f, pl = 0.0f;
    if (a.letterbox) {
        inv_s = 1.0f / a.letterbox[b * 3 + 0];
        pt = a.letterbox[b * 3 + 1];
        pl = a.letterbox[b * 3 + 2];
    }
    uint32_t gy, gx;
    L.d_W.divmod(cell, gy, gx);
    int box_an = -1, tie_seen = 0;
    float4 box = make_float4(0.f, 0.f, 0.f, 0.f);
    ml_cell<T>(a, L, b, cell, [&](int an, int c, uint32_t key) {
        bool keep = !capped || key > t;
        if (capped && key == t) keep = tie_seen++ < my_tk;
        if (!keep) return;
        if (an != box_an) {   // the row's box, exactly as yb_filter_compact builds it
            uint32_t cs;
            const T* x = reinterpret_cast<const T*>(L.pred) + ml_row(a, L, b, cell * (uint32_t)a.A + an, cs);
            float v[4], sg[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) v[k] = ldg_f(x + (size_t)k * cs);
            sigmoid_ref_batch<4>(v, sg);
            box = filter_box(a, L, sg[0], sg[1], sg[2], sg[3], gx, gy, __ldg(L.anchors + an * 2),
                             __ldg(L.anchors + an * 2 + 1), inv_s, pt, pl);
            box_an = an;
        }
        const size_t o = (size_t)b * a.cap + pos;
        a.boxes[o] = box;
        a.scores[o] = __uint_as_float(key);
        a.classes[o] = (int64_t)c;
        ++pos;
    });
}

// workspace layout, all 4-byte words: hist | state | tile_above | tile_ties | thr_above | thr_ties
static size_t ml_workspace(int B, uint32_t tiles, MlArgs* m, void* ws) {
    const size_t hist = (size_t)B * 3 * kMlBins, state = (size_t)B * ML_WORDS, tl = (size_t)B * tiles,
                 th = tl * kMlTile;
    if (m) {
        uint32_t* w = reinterpret_cast<uint32_t*>(ws);
        m->hist = w;
        m->state = reinterpret_cast<int*>(w + hist);
        m->tile_above = m->state + state;
        m->tile_ties = m->tile_above + tl;
        m->thr_above = m->tile_ties + tl;
        m->thr_ties = m->thr_above + th;
    }
    return (hist + state + 2 * tl + 2 * th) * sizeof(uint32_t);
}

template <typename T>
static int ml_launch(const yb_heads_desc* d, const FilterArgs& a, const MlArgs& m, bool may_cap, int* counts,
                     cudaStream_t st) {
    const dim3 grid(m.n.tiles_per_img, d->B);
    YB_CUDA(cudaMemsetAsync(m.hist, 0, (size_t)d->B * 3 * kMlBins * sizeof(unsigned), st));
    YB_LAUNCH("filter_ml_count_kernel", st, (filter_ml_count_kernel<T><<<grid, kMlTile, 0, st>>>(a, m)));
    YB_LAUNCH("filter_ml_select_kernel", st, (filter_ml_select_kernel<<<d->B, kMlSelect, 0, st>>>(m, 1, counts)));
    if (may_cap) {
        for (int level = 2; level <= 3; ++level) {
            YB_LAUNCH("filter_ml_refine_kernel", st, (filter_ml_refine_kernel<T><<<grid, kMlTile, 0, st>>>(a, m, level)));
            YB_LAUNCH("filter_ml_select_kernel", st, (filter_ml_select_kernel<<<d->B, kMlSelect, 0, st>>>(m, level, counts)));
        }
        YB_LAUNCH("filter_ml_refine_kernel", st, (filter_ml_refine_kernel<T><<<grid, kMlTile, 0, st>>>(a, m, 4)));
    }
    YB_LAUNCH("filter_ml_emit_kernel", st, (filter_ml_emit_kernel<T><<<grid, kMlTile, 0, st>>>(a, m)));
    return 0;
}

}  // namespace yb

extern "C" size_t yb_filter_multilabel_workspace_bytes(const yb_heads_desc* d, int max_candidates) {
    (void)max_candidates;   // the workspace does not depend on the cap
    yb::FilterArgs a;
    if (yb::filter_fill(d, "filter_multilabel", false, a, 1, yb::kMlTile)) return 0;
    const yb::FilterNchw n = yb::filter_cell_tiles(a, d->S, yb::kMlTile);
    return yb::ml_workspace(d->B, n.tiles_per_img, nullptr, nullptr);
}

extern "C" int yb_filter_multilabel(const yb_heads_desc* d, float conf_thres, const float* letterbox, int max_candidates,
                                    float* boxes, float* scores, int64_t* classes, int* counts, int* totals, int cap,
                                    void* ws, size_t ws_bytes, void* stream) {
    using namespace yb;
    FilterArgs a;
    int rc = filter_fill(d, "filter_multilabel", true, a, 1, kMlTile);
    if (rc) return rc;
    YB_CHECK_ARG(max_candidates >= 1, "filter_multilabel: max_candidates must be >= 1, got %d", max_candidates);
    unsigned long long rows = 0;
    for (int s = 0; s < d->S; ++s) rows += a.sc[s].img_rows;
    const unsigned long long pairs = rows * (unsigned long long)d->nc;
    YB_CHECK_ARG(pairs < (1ull << 31), "filter_multilabel: rows * nc too large");
    const unsigned long long need_cap = pairs < (unsigned long long)max_candidates ? pairs : (unsigned long long)max_candidates;
    YB_CHECK_ARG(cap >= 0 && (unsigned long long)cap >= need_cap, "filter_multilabel: cap %d < min(max_candidates, rows*nc) = %llu",
                 cap, need_cap);
    if (d->B == 0) return 0;
    YB_CHECK_ARG(boxes && scores && classes && counts && ws && cap > 0, "filter_multilabel: null output");
    YB_CHECK_ARG(aligned16(boxes) && (reinterpret_cast<uintptr_t>(ws) & 3u) == 0,
                 "filter_multilabel: boxes must be 16-byte, the workspace 4-byte aligned");
    if (ws_bytes < yb_filter_multilabel_workspace_bytes(d, max_candidates)) {
        set_error("filter_multilabel: workspace too small");
        return YB_EWORKSPACE;
    }
    YB_CHECK_ARG(d->B <= 65535, "filter_multilabel: B too large");
    a.cap = cap; a.conf = conf_thres; a.letterbox = letterbox;
    a.boxes = reinterpret_cast<float4*>(boxes); a.scores = scores; a.classes = classes; a.counts = counts;
    MlArgs m;
    m.n = filter_cell_tiles(a, d->S, kMlTile);
    m.K = max_candidates;
    m.totals = totals;
    ml_workspace(d->B, m.n.tiles_per_img, &m, ws);
    const bool may_cap = pairs > (unsigned long long)max_candidates;
    cudaStream_t st = (cudaStream_t)stream;
    YB_DISPATCH_DTYPE(d->dtype, T, return ml_launch<T>(d, a, m, may_cap, counts, st));
    return 0;
}
