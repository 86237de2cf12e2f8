// yb_loss.cu — K3: CIoU loss and the fused YOLO loss (forward + backward in one pass).
// Reference: ciou_loss train.py:634-710, yolo_loss :781-838, yolo_loss_multiscale :840-886.
//
// Bound: HBM.  Algorithmic bytes (SURVEY 8d):
//   A_loss = T (dense gradient write) + 2*rows*min(row_bytes,32) (objectness sectors of pred
//            and target) + 2*P*row_bytes (positive rows)
// Three launches for all scales together:
//   loss_main_kernel      every row: objectness BCE + its gradient, dense gradient tile written
//                         as coalesced float4, positive rows (target obj > 0.5) appended to a list
//   loss_positive_kernel  one warp per positive row: decode + CIoU fwd/bwd + class BCE fwd/bwd
//   loss_finalize_kernel  (after the optional all-reduce of S*4 doubles) scales the positive
//                         rows' gradients by 1/P_s and emits the four scalars
#include "yb_common.cuh"

namespace yb {

// ------------------------------------------------------------------------------------------
// CIoU for one box pair, forward value and gradients w.r.t. both boxes for upstream grad 1.
// Expression order follows train.py:646-708 line by line; alpha is a constant (:701-702).
// min/max ties split the gradient 0.5/0.5 and clamp(min=0) passes gradient at exactly 0,
// as torch autograd does.
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ float tie_lt(float a, float b) { return a < b ? 1.0f : (a == b ? 0.5f : 0.0f); }

template <bool WANT_GRAD>
__device__ __forceinline__ float ciou_pair(const float p[4], const float t[4], float eps,
                                           float gp[4], float gt[4]) {
    const float px = p[0], py = p[1], pw = p[2], ph = p[3];
    const float tx = t[0], ty = t[1], tw = t[2], th = t[3];
    const float px1 = px - pw * 0.5f, py1 = py - ph * 0.5f, px2 = px + pw * 0.5f, py2 = py + ph * 0.5f;
    const float tx1 = tx - tw * 0.5f, ty1 = ty - th * 0.5f, tx2 = tx + tw * 0.5f, ty2 = ty + th * 0.5f;

    const float ix1 = fmaxf(px1, tx1), iy1 = fmaxf(py1, ty1);
    const float ix2 = fminf(px2, tx2), iy2 = fminf(py2, ty2);
    const float iw_raw = ix2 - ix1, ih_raw = iy2 - iy1;
    const float iw = fmaxf(iw_raw, 0.0f), ih = fmaxf(ih_raw, 0.0f);
    const float inter = iw * ih;
    const float parea = pw * ph, tarea = tw * th;
    const float uni = (parea + tarea) - inter;
    const float U = uni + eps;
    const float iou = inter / U;

    const float dx = px - tx, dy = py - ty;
    const float cd = dx * dx + dy * dy;
    const float ex1 = fminf(px1, tx1), ey1 = fminf(py1, ty1);
    const float ex2 = fmaxf(px2, tx2), ey2 = fmaxf(py2, ty2);
    const float ew = ex2 - ex1, eh = ey2 - ey1;
    const float ed = (ew * ew + eh * eh) + eps;
    const float dp = cd / ed;

    const float php = ph + eps, thp = th + eps;
    const float rp = pw / php, rt = tw / thp;
    const float ap = atanf(rp), at = atanf(rt);
    const float kv = 0.40528473456935109f;  // 4 / pi^2 (python double, cast to fp32 by torch)
    const float d = ap - at;
    const float v = kv * (d * d);
    const float alpha = v / (((1.0f - iou) + v) + eps);
    const float ciou = (iou - dp) - alpha * v;
    const float loss = 1.0f - ciou;

    if (WANT_GRAD) {
        // upstream: dL/dciou = -1
        const float g_iou = -1.0f, g_dp = 1.0f, g_v = alpha;
        // iou = inter / U
        const float g_inter1 = g_iou / U;
        const float g_U = -g_iou * (iou / U);
        // U = ((parea + tarea) - inter) + eps
        const float g_parea = g_U, g_tarea = g_U;
        const float g_inter = g_inter1 - g_U;
        // inter = iw * ih ; clamp(min=0) ; iw_raw = ix2 - ix1
        const float g_iwr = (iw_raw >= 0.0f) ? g_inter * ih : 0.0f;
        const float g_ihr = (ih_raw >= 0.0f) ? g_inter * iw : 0.0f;
        // dp = cd / ed
        const float g_cd = g_dp / ed;
        const float g_ed = -g_dp * (dp / ed);
        const float g_dx = g_cd * (2.0f * dx), g_dy = g_cd * (2.0f * dy);
        const float g_ew = g_ed * (2.0f * ew), g_eh = g_ed * (2.0f * eh);
        // corner gradients: ix1 = max(p1,t1), ix2 = min(p2,t2), ex1 = min(p1,t1), ex2 = max(p2,t2)
        const float mx1 = tie_lt(tx1, px1), mx2 = tie_lt(px2, tx2);  // weight on the pred corner
        const float my1 = tie_lt(ty1, py1), my2 = tie_lt(py2, ty2);
        const float nx1 = tie_lt(px1, tx1), nx2 = tie_lt(tx2, px2);  // enclosing box: pred weight
        const float ny1 = tie_lt(py1, ty1), ny2 = tie_lt(ty2, py2);
        const float g_px1 = (-g_iwr) * mx1 + (-g_ew) * nx1;
        const float g_px2 = g_iwr * mx2 + g_ew * nx2;
        const float g_py1 = (-g_ihr) * my1 + (-g_eh) * ny1;
        const float g_py2 = g_ihr * my2 + g_eh * ny2;
        // v = kv * d^2 ; d = atan(rp) - atan(rt)
        const float g_d = g_v * (kv * (2.0f * d));
        const float g_rp = g_d / (rp * rp + 1.0f);
        gp[0] = g_dx + g_px1 + g_px2;
        gp[1] = g_dy + g_py1 + g_py2;
        gp[2] = g_parea * ph + (g_px2 - g_px1) * 0.5f + g_rp / php;
        gp[3] = g_parea * pw + (g_py2 - g_py1) * 0.5f - g_rp * (rp / php);
        if (gt) {
            const float g_tx1 = (-g_iwr) * (1.0f - mx1) + (-g_ew) * (1.0f - nx1);
            const float g_tx2 = g_iwr * (1.0f - mx2) + g_ew * (1.0f - nx2);
            const float g_ty1 = (-g_ihr) * (1.0f - my1) + (-g_eh) * (1.0f - ny1);
            const float g_ty2 = g_ihr * (1.0f - my2) + g_eh * (1.0f - ny2);
            const float g_rt = -g_d / (rt * rt + 1.0f);
            gt[0] = -g_dx + g_tx1 + g_tx2;
            gt[1] = -g_dy + g_ty1 + g_ty2;
            gt[2] = g_tarea * th + (g_tx2 - g_tx1) * 0.5f + g_rt / thp;
            gt[3] = g_tarea * tw + (g_ty2 - g_ty1) * 0.5f - g_rt * (rt / thp);
        }
    }
    return loss;
}

// ------------------------------------------------------------------------------------------
// standalone ciou_loss(pred_boxes, target_boxes, eps)  — train.py:634-710
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) ciou_kernel(const float4* __restrict__ pred,
                                                   const float4* __restrict__ tgt, long long N,
                                                   float eps, float4* __restrict__ gpred,
                                                   float4* __restrict__ gtgt,
                                                   double* __restrict__ acc) {
    const float invN = 1.0f / (float)N;
    float local = 0.0f;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < N;
         i += (long long)gridDim.x * blockDim.x) {
        float4 p4 = pred[i], t4 = tgt[i];
        float p[4] = {p4.x, p4.y, p4.z, p4.w}, t[4] = {t4.x, t4.y, t4.z, t4.w};
        float gp[4], gt[4];
        float l;
        if (gpred || gtgt) l = ciou_pair<true>(p, t, eps, gp, gtgt ? gt : nullptr);
        else l = ciou_pair<false>(p, t, eps, gp, nullptr);
        local += l;
        if (gpred) gpred[i] = make_float4(gp[0] * invN, gp[1] * invN, gp[2] * invN, gp[3] * invN);
        if (gtgt) gtgt[i] = make_float4(gt[0] * invN, gt[1] * invN, gt[2] * invN, gt[3] * invN);
    }
    __shared__ double s_part[8];
    double w = warp_sum((double)local);
    if ((threadIdx.x & 31) == 0) s_part[threadIdx.x >> 5] = w;
    __syncthreads();
    if (threadIdx.x == 0) {
        double tot = 0.0;
        for (int k = 0; k < (int)(blockDim.x >> 5); ++k) tot += s_part[k];
        atomicAdd(acc, tot);
    }
}

__global__ void ciou_mean_kernel(const double* __restrict__ acc, long long N, float* __restrict__ out) {
    // mean of an empty tensor is NaN in torch (0/0)
    out[0] = (N == 0) ? __int_as_float(0x7fc00000) : (float)(acc[0] / (double)N);
}

// ------------------------------------------------------------------------------------------
// fused multi-scale loss
// ------------------------------------------------------------------------------------------
constexpr int kTileRows = 256;  // rows per tile == threads per CTA of loss_main_kernel

struct LossScale {
    const void* pred;     // element type T of the kernels
    const float* tgt;
    const float* anchors;
    void* grad;           // fp32: written by stage 1; half: written by yb_loss_grad_emit only
    float* dobj;          // half heads: fp32 objectness gradient of every row (canonical order), else null
    const uint32_t* bits; // sparse targets: 1 bit per row (positive), else null
    uint32_t rows;        // B*H*W*A (local)
    uint32_t tile_begin;  // first global tile index of this scale
    uint32_t list_begin;  // offset of this scale's positive list in ws
    int H, W;
    float inv_w, inv_h;
    float obj_scale;      // coef_obj / (B_global*H*W*A)
    FastDiv d_A, d_W, d_H;
    // NCHW layout (f-2): pred/grad are (B, A*row, H, W); element (r, c) of canonical row r=(b,gy,gx,a)
    // lives at ((b*A + a)*row + c)*HW + gy*W + gx
    uint32_t HW, n_float;
    FastDiv d_HW;
};

struct LossArgs {
    int S, A, nc, nchw;
    uint32_t row;        // 5+nc
    uint32_t n_tiles;
    float inv_img, eps;
    FastDiv d_row;
    LossScale sc[YB_MAX_SCALES];
    int* pos_count;      // [YB_MAX_SCALES] in ws
    uint32_t* pos_list;  // ws
    int fuse_norm;               // single rank (B_global == B): the positive kernel writes final gradients
    float coef_box[YB_MAX_SCALES], coef_cls[YB_MAX_SCALES];
    const uint32_t* pos_ent;     // sparse targets: entry id of each listed row
    const SparseEntry* entries;  // sparse targets: target rows
    double* partials;    // S*4: {sum(1-ciou), n_pos, sum bce_obj, sum bce_cls}; null in the half emit pass
    const double* red;   // half emit pass: the reduced partials (P_s of the normalisation), else null
    const float* gscale; // half emit pass: upstream gradient s of `total` (device), else null
};

// offset of channel 0 of canonical row r, and the distance between its channels
__device__ __forceinline__ size_t row_base(const LossArgs& a, const LossScale& L, uint32_t r, uint32_t& cstride) {
    if (!a.nchw) {
        cstride = 1u;
        return (size_t)r * a.row;
    }
    uint32_t cellb, an, b, cell;
    L.d_A.divmod(r, cellb, an);
    L.d_HW.divmod(cellb, b, cell);
    cstride = L.HW;
    return ((size_t)(b * a.A + an) * a.row) * L.HW + cell;
}

struct LossWs {
    int pos_count[YB_MAX_SCALES];
    int pad[12];
};

template <typename T, bool SPARSE>
__global__ void __launch_bounds__(kTileRows) loss_main_kernel(const LossArgs a) {
    __shared__ float s_dobj[kTileRows];
    __shared__ float s_warp[kTileRows / 32];
    double cta_sum[YB_MAX_SCALES];
#pragma unroll
    for (int s = 0; s < YB_MAX_SCALES; ++s) cta_sum[s] = 0.0;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;

    for (uint32_t tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x) {
        int s = 0;
#pragma unroll
        for (int k = 1; k < YB_MAX_SCALES; ++k)
            if (k < a.S && tile >= a.sc[k].tile_begin) s = k;
        const LossScale& L = a.sc[s];
        const uint32_t row0 = (tile - L.tile_begin) * kTileRows;
        const uint32_t nrows = min((uint32_t)kTileRows, L.rows - row0);

        // phase 1: objectness of one row per thread (4-byte loads at a stride of one row:
        // one 32-byte sector per row of pred and of target)
        float bce = 0.0f;
        bool pos = false;
        if (threadIdx.x < nrows) {
            const size_t off = (size_t)(row0 + threadIdx.x) * a.row + 4;
            const float x = ldg_f(reinterpret_cast<const T*>(L.pred) + off);
            float t;
            if (SPARSE) {
                const uint32_t r = row0 + threadIdx.x;
                t = ((__ldg(L.bits + (r >> 5)) >> (r & 31)) & 1u) ? 1.0f : 0.0f;
            } else {
                t = __ldg(L.tgt + off);
            }
            bce = bce_logits_ref(x, t);
            const float dobj = (sigmoidf_ref(x) - t) * L.obj_scale;
            if constexpr (kHalf<T>) {   // no dense gradient here: the emit pass writes it once s is known
                if (L.dobj) L.dobj[row0 + threadIdx.x] = dobj;
            } else {
                s_dobj[threadIdx.x] = dobj;
            }
            pos = t > 0.5f;
        }
        // positives: warp-aggregated append
        const unsigned bal = SPARSE ? 0u : __ballot_sync(0xffffffffu, pos);  // sparse: lists come from the assignment
        if (bal) {
            int base = 0;
            if (lane == 0) base = atomicAdd(a.pos_count + s, __popc(bal));
            base = __shfl_sync(0xffffffffu, base, 0);
            if (pos) a.pos_list[L.list_begin + base + __popc(bal & ((1u << lane) - 1))] = row0 + threadIdx.x;
        }
        const float wsum = warp_sum(bce);
        if (lane == 0) s_warp[warp] = wsum;
        __syncthreads();
        if (threadIdx.x == 0) {
            float tsum = 0.0f;
#pragma unroll
            for (int k = 0; k < kTileRows / 32; ++k) tsum += s_warp[k];
#pragma unroll
            for (int k = 0; k < YB_MAX_SCALES; ++k)
                if (k == s) cta_sum[k] += (double)tsum;
        }
        // phase 2: dense gradient tile, coalesced float4: zeros except the objectness column
        if (!kHalf<T> && L.grad) {
            const uint32_t nfl = nrows * a.row;
            float* g = reinterpret_cast<float*>(L.grad) + (size_t)row0 * a.row;
            float4* g4 = reinterpret_cast<float4*>(g);
            const uint32_t nvec = nfl >> 2;
            for (uint32_t v = threadIdx.x; v < nvec; v += kTileRows) {
                uint32_t r, c;
                a.d_row.divmod(v * 4u, r, c);
                float o[4];
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    o[k] = (c == 4) ? s_dobj[r] : 0.0f;
                    if (++c == a.row) { c = 0; ++r; }
                }
                g4[v] = make_float4(o[0], o[1], o[2], o[3]);
            }
            if (threadIdx.x < (nfl & 3u)) {
                uint32_t e = nvec * 4u + threadIdx.x, r, c;
                a.d_row.divmod(e, r, c);
                g[e] = (c == 4) ? s_dobj[r] : 0.0f;
            }
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
#pragma unroll
        for (int s = 0; s < YB_MAX_SCALES; ++s)
            if (s < a.S && cta_sum[s] != 0.0) atomicAdd(a.partials + s * 4 + 2, cta_sum[s]);
    }
}

// NCHW variant of the main pass (f-2): walks the gradient tensor (B, A*row, H, W) as a flat float4
// stream.  84 of 85 channel planes (nc=80) are pure zero stores; an objectness plane is a coalesced
// read of the logits (4 bytes per row instead of one 128-byte DRAM line per row in the reference
// layout), the targets' objectness (dense: reference layout; sparse: the bit map) and a coalesced
// store of the gradient.
constexpr int kNchwVecs = 4;  // float4 vectors per thread and tile: 256 threads x 4 x 16 B = 16 KB per tile

template <typename T, bool SPARSE>
__device__ __forceinline__ float nchw_obj_elem(const LossArgs& a, const LossScale& L, int s, uint32_t ba, uint32_t cell,
                                               float x, float& bce) {
    uint32_t b, an;
    L.d_A.divmod(ba, b, an);
    const uint32_t r = (b * L.HW + cell) * (uint32_t)a.A + an;  // canonical row
    float t;
    if (SPARSE) t = ((__ldg(L.bits + (r >> 5)) >> (r & 31)) & 1u) ? 1.0f : 0.0f;
    else t = __ldg(L.tgt + (size_t)r * a.row + 4);
    bce += bce_logits_ref(x, t);
    if (!SPARSE && t > 0.5f) {
        const int slot = atomicAdd(a.pos_count + s, 1);
        a.pos_list[L.list_begin + slot] = r;
    }
    const float dobj = (sigmoidf_ref(x) - t) * L.obj_scale;
    if constexpr (kHalf<T>) {
        if (L.dobj) L.dobj[r] = dobj;
    }
    return dobj;
}

template <typename T, bool SPARSE>
__global__ void __launch_bounds__(kTileRows) loss_main_nchw_kernel(const LossArgs a) {
    // 4 elements per step for every element type (16-byte fp32 vectors, 8-byte half vectors): each thread sums the
    // same elements in the same order, so the half heads' loss is bit-identical to the fp32 path's
    constexpr uint32_t V = 4;
    __shared__ double s_part[kTileRows / 32][YB_MAX_SCALES];
    double acc[YB_MAX_SCALES];
#pragma unroll
    for (int s = 0; s < YB_MAX_SCALES; ++s) acc[s] = 0.0;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;

    for (uint32_t tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x) {
        int s = 0;
#pragma unroll
        for (int k = 1; k < YB_MAX_SCALES; ++k)
            if (k < a.S && tile >= a.sc[k].tile_begin) s = k;
        const LossScale& L = a.sc[s];
        float bce = 0.0f;
#pragma unroll
        for (int k = 0; k < kNchwVecs; ++k) {
            const uint32_t e0 = (((tile - L.tile_begin) * kNchwVecs + k) * kTileRows + threadIdx.x) * V;
            if (e0 >= L.n_float) continue;
            uint32_t plane, within;
            L.d_HW.divmod(e0, plane, within);
            float o[V];
#pragma unroll
            for (int j = 0; j < (int)V; ++j) o[j] = 0.0f;
            if (within + V <= L.HW && e0 + V <= L.n_float) {  // the common case: one channel plane
                uint32_t ba, c;
                a.d_row.divmod(plane, ba, c);
                if (c == 4u) {
                    if constexpr (kHalf<T>) {
                        const uint2 x2 = __ldg(reinterpret_cast<const uint2*>(reinterpret_cast<const T*>(L.pred) + e0));
                        const T* x = reinterpret_cast<const T*>(&x2);
#pragma unroll
                        for (int j = 0; j < (int)V; ++j) o[j] = nchw_obj_elem<T, SPARSE>(a, L, s, ba, within + j, to_f32(x[j]), bce);
                    } else {
                        const float4 x4 = __ldg(reinterpret_cast<const float4*>(reinterpret_cast<const T*>(L.pred) + e0));
                        o[0] = nchw_obj_elem<T, SPARSE>(a, L, s, ba, within, x4.x, bce);
                        o[1] = nchw_obj_elem<T, SPARSE>(a, L, s, ba, within + 1, x4.y, bce);
                        o[2] = nchw_obj_elem<T, SPARSE>(a, L, s, ba, within + 2, x4.z, bce);
                        o[3] = nchw_obj_elem<T, SPARSE>(a, L, s, ba, within + 3, x4.w, bce);
                    }
                }
                if (!kHalf<T> && L.grad)   // half: the emit pass writes the gradient
                    *reinterpret_cast<float4*>(reinterpret_cast<float*>(L.grad) + e0) = make_float4(o[0], o[1], o[2], o[3]);
            } else {  // a vector straddling two planes or the end of the tensor (H*W not a multiple of V)
                for (uint32_t j = 0; j < V && e0 + j < L.n_float; ++j) {
                    uint32_t ba, c;
                    a.d_row.divmod(plane, ba, c);
                    float v = 0.0f;
                    if (c == 4u) v = nchw_obj_elem<T, SPARSE>(a, L, s, ba, within, ldg_f(reinterpret_cast<const T*>(L.pred) + e0 + j), bce);
                    if (!kHalf<T> && L.grad) reinterpret_cast<float*>(L.grad)[e0 + j] = v;
                    if (++within == L.HW) { within = 0; ++plane; }
                }
            }
        }
#pragma unroll
        for (int k = 0; k < YB_MAX_SCALES; ++k)
            if (k == s) acc[k] += (double)bce;
    }
#pragma unroll
    for (int s = 0; s < YB_MAX_SCALES; ++s) {
        const double w = warp_sum(acc[s]);
        if (lane == 0) s_part[warp][s] = w;
    }
    __syncthreads();
    if (threadIdx.x < YB_MAX_SCALES && (int)threadIdx.x < a.S) {
        double tot = 0.0;
#pragma unroll
        for (int k = 0; k < kTileRows / 32; ++k) tot += s_part[k][threadIdx.x];
        if (tot != 0.0) atomicAdd(a.partials + threadIdx.x * 4 + 2, tot);
    }
}

// one warp per positive row.  Half heads run it twice: in stage 1 for the loss sums only (grad null), and in the
// emit pass (partials null, red/gscale set) for the gradient of the positive rows, fully normalised and scaled.
template <typename T, bool SPARSE>
__global__ void __launch_bounds__(256) loss_positive_kernel(const LossArgs a) {
    const int lane = threadIdx.x & 31;
    const int warps_per_cta = blockDim.x >> 5;
    const uint32_t gwarp = blockIdx.x * warps_per_cta + (threadIdx.x >> 5);
    const uint32_t nwarps = gridDim.x * warps_per_cta;
    for (int s = 0; s < a.S; ++s) {
        const LossScale& L = a.sc[s];
        const uint32_t P = (uint32_t)a.pos_count[s];
        double acc_box = 0.0, acc_cls = 0.0;
        // single rank: the local positive count IS the global one, so the normalisation that
        // loss_finalize_kernel would apply (same two roundings: unnormalised value, then * k) happens here
        float k_box = 1.0f, k_cls = 1.0f, gsc = 1.0f;
        if constexpr (kHalf<T>) {   // emit pass: the normalisation of loss_finalize_kernel, from the reduced P_s
            const double Pg = a.red ? a.red[s * 4 + 1] : 0.0;
            if (Pg > 0.0) {
                k_box = (float)((double)a.coef_box[s] / Pg);
                k_cls = a.nc > 0 ? (float)((double)a.coef_cls[s] / (Pg * (double)a.nc)) : 0.0f;
            }
            if (a.gscale) gsc = __ldg(a.gscale);
        } else if (a.fuse_norm && P > 0) {
            k_box = (float)((double)a.coef_box[s] / (double)P);
            k_cls = a.nc > 0 ? (float)((double)a.coef_cls[s] / ((double)P * (double)a.nc)) : 0.0f;
        }
        // gradient entry i of the row: fp32 as before; half: round_D((g * k) * s), the fp32 path's two roundings,
        // its scale_kernel product and the cast to the head dtype
        auto put = [&](size_t i, float g, float k) {
            if constexpr (kHalf<T>) reinterpret_cast<T*>(L.grad)[i] = from_f32<T>((g * k) * gsc);
            else reinterpret_cast<float*>(L.grad)[i] = a.fuse_norm ? g * k : g;
        };
        for (uint32_t k = gwarp; k < P; k += nwarps) {
            const uint32_t r = a.pos_list[L.list_begin + k];
            uint32_t cs;
            const size_t xb = row_base(a, L, r, cs);
            const T* x = reinterpret_cast<const T*>(L.pred) + xb;
            const float* t = SPARSE ? nullptr : L.tgt + (size_t)r * a.row;  // dense targets keep the reference layout
            SparseEntry ent = {0.f, 0.f, 0.f, 0.f, 0, 0, 0, 0};
            if (SPARSE) ent = a.entries[a.pos_ent[L.list_begin + k]];
            uint32_t cell, an, gy_b, gx, gy, bi;
            L.d_A.divmod(r, cell, an);
            L.d_W.divmod(cell, gy_b, gx);
            L.d_H.divmod(gy_b, bi, gy);
            const float aw = __ldg(L.anchors + an * 2), ah = __ldg(L.anchors + an * 2 + 1);
            const float xr[4] = {to_f32(x[0]), to_f32(x[(size_t)cs]), to_f32(x[2 * (size_t)cs]), to_f32(x[3 * (size_t)cs])};
            const float p[4] = {decode_xy(xr[0], (float)gx, L.inv_w), decode_xy(xr[1], (float)gy, L.inv_h),
                                decode_wh(xr[2], aw, a.inv_img), decode_wh(xr[3], ah, a.inv_img)};
            const float tb[4] = {SPARSE ? ent.x : t[0], SPARSE ? ent.y : t[1], SPARSE ? ent.w : t[2],
                                 SPARSE ? ent.h : t[3]};
            float gp[4];
            const float l = ciou_pair<true>(p, tb, a.eps, gp, nullptr);
            // class BCE, lanes stride over classes
            float cls = 0.0f;
            for (int c = lane; c < a.nc; c += 32) {
                const float xc = to_f32(x[(size_t)(5 + c) * cs]);
                const float tc = SPARSE ? (c == ent.cls ? 1.0f : 0.0f) : t[5 + c];
                cls += bce_logits_ref(xc, tc);
                if (L.grad) {
                    const float g = sigmoidf_ref(xc) - tc;
                    put(xb + (size_t)(5 + c) * cs, g, k_cls);
                }
            }
            cls = warp_sum(cls);
            if (L.grad && lane < 4) {
                // chain through decode (same order as decode_kernel<true>)
                const float sgm = sigmoidf_ref(xr[lane]);
                const float ds = (1.0f - sgm) * sgm;
                float g;
                if (lane < 2) {
                    g = ((gp[lane] * (lane == 0 ? L.inv_w : L.inv_h)) * 2.0f) * ds;
                } else {
                    const float anc = lane == 2 ? aw : ah;
                    const float u = 2.0f * sgm;
                    g = (((gp[lane] * (anc * a.inv_img)) * (2.0f * u)) * 2.0f) * ds;
                }
                put(xb + (size_t)lane * cs, g, k_box);
            }
            acc_box += (double)l;
            acc_cls += (double)cls;
        }
        if (!kHalf<T> || a.partials) {
            if (lane == 0 && gwarp < P) {
                atomicAdd(a.partials + s * 4 + 0, acc_box);
                if (a.nc > 0) atomicAdd(a.partials + s * 4 + 3, acc_cls);
            }
            if (gwarp == 0 && lane == 0) a.partials[s * 4 + 1] = (double)P;
        }
    }
}

struct FinalizeArgs {
    LossArgs a;
    const double* partials;  // reduced
    float* out4;
    float* per_scale;
    double n_obj[YB_MAX_SCALES];  // B_global*H*W*A
    float w_box, w_cls;
    float w_obj[YB_MAX_SCALES];
    float coef_box[YB_MAX_SCALES], coef_cls[YB_MAX_SCALES];
};

__global__ void __launch_bounds__(256) loss_finalize_kernel(const FinalizeArgs f) {
    const LossArgs& a = f.a;
    const int lane = threadIdx.x & 31;
    const int warps_per_cta = blockDim.x >> 5;
    const uint32_t gwarp = blockIdx.x * warps_per_cta + (threadIdx.x >> 5);
    const uint32_t nwarps = gridDim.x * warps_per_cta;
    for (int s = 0; s < a.S; ++s) {
        const LossScale& L = a.sc[s];
        if (!L.grad || a.fuse_norm) continue;         // fused: loss_positive_kernel already normalised
        const uint32_t P = (uint32_t)a.pos_count[s];  // local positives
        const double Pg = f.partials[s * 4 + 1];      // global positives
        if (P == 0 || Pg <= 0.0) continue;
        const float k_box = (float)((double)f.coef_box[s] / Pg);
        const float k_cls = a.nc > 0 ? (float)((double)f.coef_cls[s] / (Pg * (double)a.nc)) : 0.0f;
        for (uint32_t k = gwarp; k < P; k += nwarps) {
            uint32_t cs;
            float* g = reinterpret_cast<float*>(L.grad) + row_base(a, L, a.pos_list[L.list_begin + k], cs);
            if (lane < 4) g[(size_t)lane * cs] *= k_box;
            for (int c = lane; c < a.nc; c += 32) g[(size_t)(5 + c) * cs] *= k_cls;
        }
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        float total = 0.0f, sb = 0.0f, so = 0.0f, sc = 0.0f;
        for (int s = 0; s < a.S; ++s) {
            const double Pg = f.partials[s * 4 + 1];
            const float bbox = Pg > 0.0 ? (float)(f.partials[s * 4 + 0] / Pg) : 0.0f;
            const float obj = (float)(f.partials[s * 4 + 2] / f.n_obj[s]);
            const float cls = (Pg > 0.0 && a.nc > 0) ? (float)(f.partials[s * 4 + 3] / (Pg * (double)a.nc)) : 0.0f;
            // train.py:879: 0.05 * bbox + obj_weight * obj + 0.5 * cls, accumulated in order
            const float weighted = (f.w_box * bbox + f.w_obj[s] * obj) + f.w_cls * cls;
            total += weighted; sb += bbox; so += obj; sc += cls;
            if (f.per_scale) {
                f.per_scale[s * 3 + 0] = bbox;
                f.per_scale[s * 3 + 1] = obj;
                f.per_scale[s * 3 + 2] = cls;
            }
        }
        f.out4[0] = total; f.out4[1] = sb; f.out4[2] = so; f.out4[3] = sc;
    }
}

__global__ void __launch_bounds__(256) scale_kernel(float* __restrict__ x, long long n,
                                                    const float* __restrict__ factor) {
    const float f = __ldg(factor);
    if (f == 1.0f) return;  // loss.backward(): nothing to do, no traffic
    const long long nvec = n >> 2;
    float4* x4 = reinterpret_cast<float4*>(x);
    for (long long v = blockIdx.x * (long long)blockDim.x + threadIdx.x; v < nvec;
         v += (long long)gridDim.x * blockDim.x) {
        float4 q = x4[v];
        q.x *= f; q.y *= f; q.z *= f; q.w *= f;
        x4[v] = q;
    }
    if (blockIdx.x == 0 && threadIdx.x < (n & 3)) x[nvec * 4 + threadIdx.x] *= f;
}

// Half heads, backward: the dense gradient of every scale, zeros except the objectness channel, which is
// round_D(dobj * s) (dobj: stage 1's fp32 value).  16-byte vector stores; loss_positive_kernel<T> overwrites the
// box and class channels of the positive rows afterwards.  Zeros are 0 * s, as the fp32 path's scale_kernel gives.
template <typename T>
__global__ void __launch_bounds__(256) loss_grad_emit_kernel(const LossArgs a) {
    constexpr uint32_t V = kVec<T>;
    const float gsc = __ldg(a.gscale);
    const float zero = 0.0f * gsc;
    const uint32_t tid = blockIdx.x * blockDim.x + threadIdx.x, stride = gridDim.x * blockDim.x;
    for (int s = 0; s < a.S; ++s) {
        const LossScale& L = a.sc[s];
        T* grad = reinterpret_cast<T*>(L.grad);
        if (!grad) continue;
        const float* dobj = L.dobj;
        const uint32_t n = L.n_float, nv = (n + V - 1) / V;
        for (uint32_t v = tid; v < nv; v += stride) {
            const uint32_t e0 = v * V;
            float o[V];
            if (!a.nchw) {
                uint32_t r, c;
                a.d_row.divmod(e0, r, c);
#pragma unroll
                for (int j = 0; j < (int)V; ++j) {
                    o[j] = (c == 4u && e0 + j < n) ? dobj[r] * gsc : zero;
                    if (++c == a.row) { c = 0; ++r; }
                }
            } else {
                uint32_t plane, within, ba, c;
                L.d_HW.divmod(e0, plane, within);
                a.d_row.divmod(plane, ba, c);
#pragma unroll
                for (int j = 0; j < (int)V; ++j) {
                    o[j] = zero;
                    if (c == 4u && e0 + j < n) {
                        uint32_t b, an;
                        L.d_A.divmod(ba, b, an);
                        o[j] = dobj[(b * L.HW + within) * (uint32_t)a.A + an] * gsc;
                    }
                    if (++within == L.HW) {
                        within = 0;
                        if (++c == a.row) { c = 0; ++ba; }
                    }
                }
            }
            if (e0 + V <= n) {
                *reinterpret_cast<float4*>(grad + e0) = pack16<T>(o);
            } else {
                for (uint32_t j = 0; e0 + j < n; ++j) grad[e0 + j] = from_f32<T>(o[j]);
            }
        }
    }
}

// ---- host side ----------------------------------------------------------------------------
static int loss_validate(const yb_loss_desc* d, bool need_ptrs, bool sparse = false) {
    YB_CHECK_ARG(d, "loss: null descriptor");
    YB_CHECK_ARG(d->S >= 1 && d->S <= YB_MAX_SCALES, "loss: S=%d out of range", d->S);
    YB_CHECK_ARG(d->B >= 0 && d->A > 0 && d->A <= YB_MAX_ANCHORS && d->nc >= 0, "loss: bad B/A/nc");
    YB_CHECK_ARG(d->B_global >= d->B, "loss: B_global < B");
    YB_CHECK_ARG(d->layout == YB_LAYOUT_BHWAC || d->layout == YB_LAYOUT_NCHW, "loss: unknown layout %d", d->layout);
    YB_CHECK_ARG(d->dtype == YB_DTYPE_F32 || d->dtype == YB_DTYPE_BF16 || d->dtype == YB_DTYPE_F16,
                 "loss: unknown dtype %d", d->dtype);
    unsigned long long tot = 0;
    for (int s = 0; s < d->S; ++s) {
        YB_CHECK_ARG(d->H[s] > 0 && d->W[s] > 0, "loss: bad grid at scale %d", s);
        unsigned long long n = (unsigned long long)d->B * d->H[s] * d->W[s] * d->A * (5 + d->nc);
        YB_CHECK_ARG(n < (1ull << 32), "loss: scale %d too large", s);
        tot += (unsigned long long)d->B * d->H[s] * d->W[s] * d->A;
        if (need_ptrs && d->B > 0) {
            YB_CHECK_ARG(d->pred[s] && (sparse || d->tgt[s]) && d->anchors[s], "loss: null tensor at scale %d", s);
            YB_CHECK_ARG(aligned16(d->pred[s]) && (sparse || aligned16(d->tgt[s])) && aligned16(d->grad[s]),
                         "loss: tensors must be 16-byte aligned");
        }
    }
    YB_CHECK_ARG(tot < (1ull << 32), "loss: too many rows");
    return 0;
}

static size_t loss_rows(const yb_loss_desc* d) {
    size_t rows = 0;
    for (int s = 0; s < d->S; ++s) rows += (size_t)d->B * d->H[s] * d->W[s] * d->A;
    return rows;
}
// half heads: the fp32 objectness gradient (rows floats) follows the positive list in the workspace
static size_t dobj_offset(const yb_loss_desc* d) { return (sizeof(LossWs) + loss_rows(d) * sizeof(uint32_t) + 15) / 16 * 16; }
static size_t dobj_bytes(const yb_loss_desc* d) { return d->dtype == YB_DTYPE_F32 ? 0 : loss_rows(d) * sizeof(float); }

static void loss_fill_args(const yb_loss_desc* d, void* ws, LossArgs& a) {
    const bool half = d->dtype != YB_DTYPE_F32;
    a.S = d->S; a.A = d->A; a.nc = d->nc; a.row = 5 + d->nc;
    a.nchw = d->layout == YB_LAYOUT_NCHW ? 1 : 0;
    a.inv_img = 1.0f / d->img_size; a.eps = d->eps;
    a.d_row = FastDiv(a.row);
    LossWs* w = reinterpret_cast<LossWs*>(ws);
    a.pos_count = w->pos_count;
    a.pos_list = reinterpret_cast<uint32_t*>(w + 1);
    uint32_t tile = 0, list = 0;
    for (int s = 0; s < d->S; ++s) {
        LossScale& L = a.sc[s];
        L.pred = d->pred[s]; L.tgt = d->tgt[s]; L.anchors = d->anchors[s];
        L.grad = half ? nullptr : d->grad[s];   // half: only yb_loss_grad_emit writes the gradient
        L.dobj = half ? reinterpret_cast<float*>(reinterpret_cast<char*>(ws) + dobj_offset(d)) + list : nullptr;
        L.bits = nullptr;
        L.rows = (uint32_t)((unsigned long long)d->B * d->H[s] * d->W[s] * d->A);
        L.tile_begin = tile; L.list_begin = list;
        L.HW = (uint32_t)d->H[s] * (uint32_t)d->W[s];
        L.n_float = L.rows * a.row;
        L.d_HW = FastDiv(L.HW);
        // reference layout: one tile = kTileRows rows; NCHW: one tile = kTileRows*kNchwVecs steps of 4 elements of the
        // flat tensor
        tile += a.nchw ? (L.n_float + kTileRows * 4 * kNchwVecs - 1) / (kTileRows * 4 * kNchwVecs)
                       : (L.rows + kTileRows - 1) / kTileRows;
        list += L.rows;
        L.H = d->H[s]; L.W = d->W[s];
        L.inv_w = 1.0f / (float)d->W[s]; L.inv_h = 1.0f / (float)d->H[s];
        double n_obj = (double)d->B_global * d->H[s] * d->W[s] * d->A;
        L.obj_scale = (float)((double)d->coef_obj[s] / n_obj);
        L.d_A = FastDiv(d->A); L.d_W = FastDiv(d->W[s]); L.d_H = FastDiv(d->H[s]);
    }
    a.n_tiles = tile;
    a.pos_ent = nullptr;
    a.entries = nullptr;
    a.fuse_norm = d->B_global == (long long)d->B ? 1 : 0;
    a.partials = nullptr;
    a.red = nullptr;
    a.gscale = nullptr;
    for (int s = 0; s < d->S; ++s) { a.coef_box[s] = d->coef_box[s]; a.coef_cls[s] = d->coef_cls[s]; }
}

// sparse-target workspace: [dense-layout workspace][pos_ent: rows u32][entries][bits]; the dense-layout part holds
// the objectness gradient of half heads, so pos_ent and entries do not depend on max_gt
struct SparseLayout { size_t pos_ent, entries, bits, total; uint32_t bits_begin[YB_MAX_SCALES]; };
static SparseLayout sparse_layout(const yb_loss_desc* d, int max_gt) {
    SparseLayout L;
    size_t rows = 0, words = 0;
    for (int s = 0; s < d->S; ++s) {
        const size_t r = (size_t)d->B * d->H[s] * d->W[s] * d->A;
        L.bits_begin[s] = (uint32_t)words;
        words += (r + 31) / 32;
        rows += r;
    }
    size_t o = (dobj_offset(d) + dobj_bytes(d) + 15) / 16 * 16;
    L.pos_ent = o; o = (o + rows * sizeof(uint32_t) + 15) / 16 * 16;
    L.entries = o; o += (size_t)d->B * (max_gt > 0 ? max_gt : 1) * sizeof(SparseEntry);
    L.bits = o; o += (words + 4) * sizeof(uint32_t);
    L.total = o + 16;
    return L;
}

}  // namespace yb

extern "C" size_t yb_ciou_scratch_bytes(long long) { return 16; }

extern "C" int yb_ciou_fwd_bwd(const float* pred_boxes, const float* tgt_boxes, long long N,
                               float eps, float* loss_out, float* grad_pred, float* grad_tgt,
                               void* scratch, size_t scratch_bytes, void* stream) {
    using namespace yb;
    YB_CHECK_ARG(N >= 0 && loss_out && scratch, "ciou: bad arguments");
    YB_CHECK_ARG(scratch_bytes >= 16, "ciou: scratch too small");
    YB_CHECK_ARG(N == 0 || (pred_boxes && tgt_boxes), "ciou: null boxes");
    YB_CHECK_ARG(aligned16(pred_boxes) && aligned16(tgt_boxes) && aligned16(grad_pred) && aligned16(grad_tgt),
                 "ciou: tensors must be 16-byte aligned");
    cudaStream_t st = (cudaStream_t)stream;
    double* acc = reinterpret_cast<double*>(scratch);
    YB_CUDA(cudaMemsetAsync(acc, 0, sizeof(double), st));
    if (N > 0) {
        long long want = (N + 255) / 256, cap = (long long)sm_count() * 8;
        int blocks = (int)(want < cap ? want : cap);
        YB_LAUNCH("ciou_kernel", st,
                  ciou_kernel<<<blocks, 256, 0, st>>>(reinterpret_cast<const float4*>(pred_boxes),
                                                      reinterpret_cast<const float4*>(tgt_boxes), N, eps,
                                                      reinterpret_cast<float4*>(grad_pred),
                                                      reinterpret_cast<float4*>(grad_tgt), acc));
    }
    YB_LAUNCH("ciou_mean_kernel", st, ciou_mean_kernel<<<1, 1, 0, st>>>(acc, N, loss_out));
    return 0;
}

extern "C" size_t yb_loss_workspace_bytes(const yb_loss_desc* d) {
    if (!d || d->S < 1 || d->S > YB_MAX_SCALES) return 0;
    if (d->dtype != YB_DTYPE_F32) return yb::dobj_offset(d) + yb::dobj_bytes(d) + 16;
    return sizeof(yb::LossWs) + yb::loss_rows(d) * sizeof(uint32_t) + 16;
}

namespace yb {
template <typename T, bool SPARSE>
static int loss_stage1_launch(const LossArgs& a, cudaStream_t st) {
    const int sms = sm_count();
    int blocks = (int)(a.n_tiles < (uint32_t)(sms * 8) ? a.n_tiles : (uint32_t)(sms * 8));
    if (a.nchw) YB_LAUNCH("loss_main_nchw_kernel", st, (loss_main_nchw_kernel<T, SPARSE><<<blocks, kTileRows, 0, st>>>(a)));
    else YB_LAUNCH("loss_main_kernel", st, (loss_main_kernel<T, SPARSE><<<blocks, kTileRows, 0, st>>>(a)));
    YB_LAUNCH("loss_positive_kernel", st, (loss_positive_kernel<T, SPARSE><<<sms * 2, 256, 0, st>>>(a)));
    return 0;
}
}  // namespace yb

extern "C" int yb_loss_partials(const yb_loss_desc* d, double* partials, void* ws, size_t ws_bytes,
                                void* stream) {
    using namespace yb;
    int rc = loss_validate(d, true);
    if (rc) return rc;
    YB_CHECK_ARG(partials && ws, "loss: null partials/workspace");
    if (ws_bytes < yb_loss_workspace_bytes(d)) {
        set_error("loss: workspace %zu < %zu", ws_bytes, yb_loss_workspace_bytes(d));
        return YB_EWORKSPACE;
    }
    cudaStream_t st = (cudaStream_t)stream;
    LossArgs a;
    loss_fill_args(d, ws, a);
    a.partials = partials;
    YB_CUDA(cudaMemsetAsync(ws, 0, sizeof(LossWs), st));
    YB_CUDA(cudaMemsetAsync(partials, 0, sizeof(double) * 4 * d->S, st));
    if (a.n_tiles == 0) return 0;
    YB_DISPATCH_DTYPE(d->dtype, T, return loss_stage1_launch<T, false>(a, st));
    return 0;
}

extern "C" size_t yb_loss_sparse_workspace_bytes(const yb_loss_desc* d, int max_gt) {
    if (!d || d->S < 1 || d->S > YB_MAX_SCALES || max_gt < 0) return 0;
    return yb::sparse_layout(d, max_gt).total;
}

extern "C" int yb_loss_partials_sparse(const yb_loss_desc* d, const double* labels, const int* n_gt,
                                       const double* letterbox, const float* anchors_all, int max_gt,
                                       int assign_img_size, int* status, double* partials, void* ws,
                                       size_t ws_bytes, void* stream) {
    using namespace yb;
    int rc = loss_validate(d, true, true);
    if (rc) return rc;
    YB_CHECK_ARG(partials && ws && n_gt && letterbox && anchors_all && max_gt >= 0 && (max_gt == 0 || labels) &&
                     assign_img_size > 0,
                 "loss(sparse): bad arguments");
    const SparseLayout SL = sparse_layout(d, max_gt);
    if (ws_bytes < SL.total) {
        set_error("loss(sparse): workspace %zu < %zu", ws_bytes, SL.total);
        return YB_EWORKSPACE;
    }
    cudaStream_t st = (cudaStream_t)stream;
    LossArgs a;
    loss_fill_args(d, ws, a);
    a.partials = partials;
    char* w = reinterpret_cast<char*>(ws);
    SparseOut o;
    o.entries = reinterpret_cast<SparseEntry*>(w + SL.entries);
    o.bits = reinterpret_cast<uint32_t*>(w + SL.bits);
    o.pos_count = a.pos_count;
    o.pos_list = a.pos_list;
    o.pos_ent = reinterpret_cast<uint32_t*>(w + SL.pos_ent);
    int G[YB_MAX_SCALES];
    for (int s = 0; s < d->S; ++s) {
        YB_CHECK_ARG(d->H[s] == d->W[s], "loss(sparse): the reference assigns on square grids (scale %d)", s);
        G[s] = d->H[s];
        o.bits_begin[s] = SL.bits_begin[s];
        o.list_begin[s] = a.sc[s].list_begin;
        a.sc[s].bits = o.bits + SL.bits_begin[s];
    }
    a.pos_ent = o.pos_ent;
    a.entries = o.entries;
    YB_CUDA(cudaMemsetAsync(ws, 0, sizeof(LossWs), st));
    YB_CUDA(cudaMemsetAsync(o.bits, 0, SL.total - 16 - SL.bits, st));
    YB_CUDA(cudaMemsetAsync(partials, 0, sizeof(double) * 4 * d->S, st));
    if (a.n_tiles == 0) return 0;
    rc = launch_assign_sparse(labels, n_gt, letterbox, anchors_all, d->B, max_gt, d->S, G, d->A, d->nc, assign_img_size,
                              status, o, st);
    if (rc) return rc;
    YB_DISPATCH_DTYPE(d->dtype, T, return loss_stage1_launch<T, true>(a, st));
    return 0;
}

extern "C" int yb_loss_finalize(const yb_loss_desc* d, const double* partials, float* out4,
                                float* per_scale, void* ws, size_t ws_bytes, void* stream) {
    using namespace yb;
    int rc = loss_validate(d, false);
    if (rc) return rc;
    YB_CHECK_ARG(partials && out4 && ws, "loss_finalize: null pointer");
    if (ws_bytes < yb_loss_workspace_bytes(d)) {
        set_error("loss_finalize: workspace too small");
        return YB_EWORKSPACE;
    }
    FinalizeArgs f;
    loss_fill_args(d, ws, f.a);
    f.a.partials = nullptr;
    f.partials = partials; f.out4 = out4; f.per_scale = per_scale;
    f.w_box = d->w_box; f.w_cls = d->w_cls;
    bool any_grad = false;
    for (int s = 0; s < d->S; ++s) {
        f.n_obj[s] = (double)d->B_global * d->H[s] * d->W[s] * d->A;
        f.w_obj[s] = d->w_obj[s];
        f.coef_box[s] = d->coef_box[s];
        f.coef_cls[s] = d->coef_cls[s];
        any_grad |= f.a.sc[s].grad != nullptr;
    }
    const int blocks = (any_grad && f.a.n_tiles > 0 && !f.a.fuse_norm) ? sm_count() : 1;
    cudaStream_t st = (cudaStream_t)stream;
    YB_LAUNCH("loss_finalize_kernel", st, loss_finalize_kernel<<<blocks, 256, 0, st>>>(f));
    return 0;
}

namespace yb {
template <typename T>
static int loss_emit_launch(const LossArgs& a, bool sparse, cudaStream_t st) {
    const int sms = sm_count();
    YB_LAUNCH("loss_grad_emit_kernel", st, loss_grad_emit_kernel<T><<<sms * 8, 256, 0, st>>>(a));
    if (sparse) YB_LAUNCH("loss_positive_kernel", st, (loss_positive_kernel<T, true><<<sms * 2, 256, 0, st>>>(a)));
    else YB_LAUNCH("loss_positive_kernel", st, (loss_positive_kernel<T, false><<<sms * 2, 256, 0, st>>>(a)));
    return 0;
}
}  // namespace yb

extern "C" int yb_loss_grad_emit(const yb_loss_desc* d, const double* partials, const float* grad_scale, int max_gt,
                                 void* ws, size_t ws_bytes, void* stream) {
    using namespace yb;
    const bool sparse = max_gt >= 0;
    int rc = loss_validate(d, true, sparse);
    if (rc) return rc;
    YB_CHECK_ARG(d->dtype != YB_DTYPE_F32, "loss_grad_emit: fp32 heads get their gradient from yb_loss_partials");
    YB_CHECK_ARG(partials && grad_scale && ws, "loss_grad_emit: null pointer");
    const size_t need = sparse ? yb_loss_sparse_workspace_bytes(d, max_gt) : yb_loss_workspace_bytes(d);
    if (ws_bytes < need) {
        set_error("loss_grad_emit: workspace %zu < %zu", ws_bytes, need);
        return YB_EWORKSPACE;
    }
    LossArgs a;
    loss_fill_args(d, ws, a);
    bool any = false;
    for (int s = 0; s < d->S; ++s) {
        a.sc[s].grad = d->grad[s];
        any |= d->grad[s] != nullptr;
    }
    if (!any || a.n_tiles == 0) return 0;
    a.red = partials;
    a.gscale = grad_scale;
    if (sparse) {
        const SparseLayout SL = sparse_layout(d, max_gt);
        a.pos_ent = reinterpret_cast<const uint32_t*>(reinterpret_cast<const char*>(ws) + SL.pos_ent);
        a.entries = reinterpret_cast<const SparseEntry*>(reinterpret_cast<const char*>(ws) + SL.entries);
    }
    cudaStream_t st = (cudaStream_t)stream;
    YB_DISPATCH_DTYPE(d->dtype, T, if constexpr (kHalf<T>) return loss_emit_launch<T>(a, sparse, st));
    return 0;
}

extern "C" int yb_scale_inplace(float* x, long long n, const float* factor, void* stream) {
    using namespace yb;
    YB_CHECK_ARG(n >= 0 && factor && (n == 0 || x) && aligned16(x), "scale: bad arguments");
    if (n == 0) return 0;
    long long want = (n / 4 + 255) / 256, cap = (long long)sm_count() * 8;
    int blocks = (int)(want < 1 ? 1 : (want < cap ? want : cap));
    cudaStream_t st = (cudaStream_t)stream;
    YB_LAUNCH("scale_kernel", st, scale_kernel<<<blocks, 256, 0, st>>>(x, n, factor));
    return 0;
}
