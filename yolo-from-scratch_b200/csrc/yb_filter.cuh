// yb_filter.cuh — what the single-label candidate filter (yb_filter.cu) and the multi-label one (yb_filter_ml.cu)
// share: the heads descriptor as the kernels see it, the NCHW cell tiling and the box of a row.
#pragma once
#include "yb_common.cuh"

namespace yb {

struct FilterScale : HeadScale {
    uint32_t tile_begin;   // first tile (within an image) of this scale
    uint32_t group_begin;  // first group (within an image) of this scale
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

// Box of one row from the sigmoids s0..s3 of its box logits (train.py:1154-1213): decode with the model's img_size,
// pixels, corners, letterbox reverse.  inv_s, pt, pl are the image's letterbox (ignored when a.letterbox is null).
__device__ __forceinline__ float4 filter_box(const FilterArgs& a, const FilterScale& L, float s0, float s1, float s2,
                                             float s3, uint32_t gx, uint32_t gy, float aw, float ah, float inv_s,
                                             float pt, float pl) {
    // decode (:1154) with the model's img_size
    const float bx = box_xy(s0, (float)gx, L.inv_w);
    const float by = box_xy(s1, (float)gy, L.inv_h);
    const float bw = box_wh(s2, aw, a.inv_img);
    const float bh = box_wh(s3, ah, a.inv_img);
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
        t += (a.sc[s].HW + tile_cells - 1) / tile_cells;
    }
    n.tiles_per_img = t;
    return n;
}

// Checks the descriptor (need_ptrs: pred and anchors are read) and fills everything of `a` that depends on it alone.
// G = tiles of kTileRows rows per group.
static inline int filter_fill(const yb_heads_desc* d, const char* who, bool need_ptrs, FilterArgs& a, int G,
                              uint32_t kTileRows) {
    YB_CHECK_ARG(d, "%s: null descriptor", who);
    const int rc = heads_check(*d, who, 1, true, true, need_ptrs);   // nc >= 1: train.py:1184-1189
    if (rc) return rc;
    a.S = d->S; a.A = d->A; a.nc = d->nc; a.row = 5 + d->nc;
    a.nchw = d->layout == YB_LAYOUT_NCHW ? 1 : 0;
    a.img = d->img_size; a.inv_img = 1.0f / d->img_size;
    a.G = G;
    uint32_t tile = 0, group = 0;
    for (int s = 0; s < d->S; ++s) {
        FilterScale& L = a.sc[s];
        head_scale_fill(L, *d, s);
        L.tile_begin = tile;
        L.group_begin = group;
        const uint32_t nt = (L.img_rows + kTileRows - 1) / kTileRows;
        tile += nt;
        group += (nt + a.G - 1) / a.G;
    }
    a.tiles_per_img = tile;
    a.groups_per_img = group;
    return 0;
}

}  // namespace yb
