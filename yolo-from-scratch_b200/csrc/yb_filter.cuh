// yb_filter.cuh — what the single-label candidate filter (yb_filter.cu) and the multi-label one (yb_filter_ml.cu)
// share: the heads descriptor as the kernels see it, the layout addressing, the NCHW cell tiling and the box of a row.
#pragma once
#include "yb_common.cuh"

namespace yb {

struct FilterScale {
    const void* pred;      // element type T of the kernels
    const float* anchors;
    uint32_t rows;         // rows per image at this scale = H*W*A
    uint32_t hw;           // H*W
    uint32_t tile_begin;   // first tile (within an image) of this scale
    uint32_t group_begin;  // first group (within an image) of this scale
    float inv_w, inv_h;
    FastDiv d_A, d_W;
};

struct FilterArgs {
    int S, A, nc, cap, G, nchw;
    uint32_t row, tiles_per_img, groups_per_img;
    float img, inv_img, conf;
    float obj_lo, obj_hi;      // logits clearly below / above logit(conf): sigmoid(x) > conf decided without the sigmoid
    int stage_ok;              // shared-memory staging available for this row length
    uint32_t sobj_offset;      // float offset of the sigmoid(obj) scratch in dynamic shared memory
    const float* letterbox;    // (B,3) scale, pad_top, pad_left or null
    FilterScale sc[YB_MAX_SCALES];
    int* tile_counts;          // (B, tiles_per_img)      (NCHW two-launch path)
    unsigned long long* lb_state;  // (B, groups_per_img): flag << 32 | value, zeroed before the launch
    unsigned int* lb_ticket;       // (B): next group id of every image
    unsigned int* lb_seen;         // [2]: rows / candidates of the groups that have finished their objectness pass
    float4* boxes;
    float* scores;
    int64_t* classes;
    int* counts;
};

// float offset of channel 0 of row r (within image b, scale L) and the distance between its channels;
// NCHW (f-2): the head conv's own output (B, A*row, H, W)
__device__ __forceinline__ size_t frow_base(const FilterArgs& a, const FilterScale& L, uint32_t b, uint32_t r,
                                            uint32_t& cstride) {
    if (!a.nchw) {
        cstride = 1u;
        return ((size_t)b * L.rows + r) * a.row;
    }
    uint32_t cell, an;
    L.d_A.divmod(r, cell, an);
    const uint32_t HW = L.hw;
    cstride = HW;
    return ((size_t)(b * (uint32_t)a.A + an) * a.row) * HW + cell;
}

// Box of one row from the sigmoids s0..s3 of its box logits (train.py:1154-1213): decode with the model's img_size,
// pixels, corners, letterbox reverse.  inv_s, pt, pl are the image's letterbox (ignored when a.letterbox is null).
__device__ __forceinline__ float4 filter_box(const FilterArgs& a, const FilterScale& L, float s0, float s1, float s2,
                                             float s3, uint32_t gx, uint32_t gy, float aw, float ah, float inv_s,
                                             float pt, float pl) {
    // decode (:1154) with the model's img_size
    const float bx = decode_xy_s(s0, (float)gx, L.inv_w);
    const float by = decode_xy_s(s1, (float)gy, L.inv_h);
    const float bw = decode_wh_s(s2, aw, a.inv_img);
    const float bh = decode_wh_s(s3, ah, a.inv_img);
    // pixels, corners, letterbox reverse (:1192-1213)
    const float xc = bx * a.img, yc = by * a.img, wp = bw * a.img, hp = bh * a.img;
    float x1 = xc - wp * 0.5f, y1 = yc - hp * 0.5f, x2 = xc + wp * 0.5f, y2 = yc + hp * 0.5f;
    if (a.letterbox) {
        x1 = (x1 - pl) * inv_s; y1 = (y1 - pt) * inv_s;
        x2 = (x2 - pl) * inv_s; y2 = (y2 - pt) * inv_s;
    }
    return make_float4(x1, y1, x2, y2);
}

// Cell tiling (both filters' NCHW kernels, every multi-label kernel): a tile is kFTile consecutive cells of one scale
// with all A anchors, so that thread <-> cell and the candidate order stays the canonical (cell, anchor) order.
struct FilterNchw {
    uint32_t tile_begin[YB_MAX_SCALES];  // first cell tile (within an image) of each scale
    uint32_t tiles_per_img;
};

__device__ __forceinline__ int nchw_tile_scale(const FilterArgs& a, const FilterNchw& n, uint32_t tile) {
    int s = 0;
#pragma unroll
    for (int k = 1; k < YB_MAX_SCALES; ++k)
        if (k < a.S && tile >= n.tile_begin[k]) s = k;
    return s;
}

static inline FilterNchw filter_cell_tiles(const FilterArgs& a, int S, uint32_t tile_cells) {
    FilterNchw n;
    uint32_t t = 0;
    for (int s = 0; s < S; ++s) {
        n.tile_begin[s] = t;
        t += (a.sc[s].hw + tile_cells - 1) / tile_cells;
    }
    n.tiles_per_img = t;
    return n;
}

// Checks the descriptor and fills everything of `a` that depends on it alone.  G = tiles of kTileRows rows per group.
static inline int filter_fill(const yb_heads_desc* d, FilterArgs& a, int G, uint32_t kTileRows) {
    YB_CHECK_ARG(d, "filter: null descriptor");
    YB_CHECK_ARG(d->S >= 1 && d->S <= YB_MAX_SCALES && d->B >= 0 && d->A > 0 && d->A <= YB_MAX_ANCHORS && d->nc >= 1,
                 "filter: bad S/B/A/nc (nc must be >= 1, train.py:1184-1189)");
    a.S = d->S; a.A = d->A; a.nc = d->nc; a.row = 5 + d->nc;
    YB_CHECK_ARG(d->layout == YB_LAYOUT_BHWAC || d->layout == YB_LAYOUT_NCHW, "filter: unknown layout %d", d->layout);
    YB_CHECK_ARG(d->dtype == YB_DTYPE_F32 || d->dtype == YB_DTYPE_BF16 || d->dtype == YB_DTYPE_F16,
                 "filter: unknown dtype %d", d->dtype);
    a.nchw = d->layout == YB_LAYOUT_NCHW ? 1 : 0;
    a.img = d->img_size; a.inv_img = 1.0f / d->img_size;
    a.G = G;
    uint32_t tile = 0, group = 0;
    for (int s = 0; s < d->S; ++s) {
        YB_CHECK_ARG(d->H[s] > 0 && d->W[s] > 0, "filter: bad grid at scale %d", s);
        unsigned long long n = (unsigned long long)d->B * d->H[s] * d->W[s] * d->A * (5 + d->nc);
        YB_CHECK_ARG(n < (1ull << 32), "filter: scale %d too large", s);
        FilterScale& L = a.sc[s];
        L.pred = d->pred[s]; L.anchors = d->anchors[s];
        L.rows = (uint32_t)d->H[s] * d->W[s] * d->A;
        L.hw = (uint32_t)d->H[s] * d->W[s];
        L.tile_begin = tile;
        L.group_begin = group;
        const uint32_t nt = (L.rows + kTileRows - 1) / kTileRows;
        tile += nt;
        group += (nt + a.G - 1) / a.G;
        L.inv_w = 1.0f / (float)d->W[s]; L.inv_h = 1.0f / (float)d->H[s];
        L.d_A = FastDiv(d->A); L.d_W = FastDiv(d->W[s]);
    }
    a.tiles_per_img = tile;
    a.groups_per_img = group;
    return 0;
}

}  // namespace yb
