// yb_eval.cu — f-1 (SURVEY 8f): the detection counting of eval_epoch as one kernel.
// Reference: train.py:993-1024 (decode with the default img_size, sigmoid(obj), the 4-deep python
// loop with two .item() per anchor) and compute_box_iou train.py:928-958.
//
// The reference spends 2*rows host synchronisations per batch here (rows = B*25,200 at 640^2);
// this is one pass over the objectness columns of predictions and targets plus the box columns of
// the rows where both are "on".  Bound: HBM, rows * 2 * (one DRAM line of pred and of target).
// Counts are exact integers: (TP, FP, FN) added to three int64 counters.
#include "yb_common.cuh"

namespace yb {

struct EvalScale : HeadScale {   // pred: fp32
    const float* tgt;
    uint32_t row_begin;
};

struct EvalArgs {
    int S, A;
    uint32_t row, total_rows;
    float inv_img, iou_thr;
    double conf;
    EvalScale sc[YB_MAX_SCALES];
    unsigned long long* counts;  // TP, FP, FN
};

// compute_box_iou(box1, box2) on xywh boxes, fp32, expression order of train.py:934-957
__device__ __forceinline__ float box_iou_xywh(const float a[4], const float b[4]) {
    const float ax1 = a[0] - a[2] / 2.0f, ay1 = a[1] - a[3] / 2.0f, ax2 = a[0] + a[2] / 2.0f, ay2 = a[1] + a[3] / 2.0f;
    const float bx1 = b[0] - b[2] / 2.0f, by1 = b[1] - b[3] / 2.0f, bx2 = b[0] + b[2] / 2.0f, by2 = b[1] + b[3] / 2.0f;
    const float ix1 = fmaxf(ax1, bx1), iy1 = fmaxf(ay1, by1);
    const float ix2 = fminf(ax2, bx2), iy2 = fminf(ay2, by2);
    const float inter = fmaxf(ix2 - ix1, 0.0f) * fmaxf(iy2 - iy1, 0.0f);
    const float area_a = (ax2 - ax1) * (ay2 - ay1);
    const float area_b = (bx2 - bx1) * (by2 - by1);
    const float uni = (area_a + area_b) - inter;
    return inter / (uni + 1e-6f);
}

constexpr int kEvalThreads = 256;
constexpr int kEvalIlp = 4;

__global__ void __launch_bounds__(kEvalThreads) eval_count_kernel(const EvalArgs a) {
    __shared__ unsigned int s_cnt[3];
    if (threadIdx.x < 3) s_cnt[threadIdx.x] = 0u;
    __syncthreads();
    unsigned int tp = 0, fp = 0, fn = 0;
    const uint32_t stride = gridDim.x * kEvalThreads;
    for (uint32_t g0 = blockIdx.x * kEvalThreads + threadIdx.x; g0 < a.total_rows; g0 += stride * kEvalIlp) {
        float xo[kEvalIlp], to[kEvalIlp];
        const float *px[kEvalIlp], *pt[kEvalIlp];
        int sidx[kEvalIlp];
        uint32_t rr[kEvalIlp];
#pragma unroll
        for (int u = 0; u < kEvalIlp; ++u) {
            const uint32_t g = g0 + (uint32_t)u * stride;
            xo[u] = 0.0f; to[u] = 0.0f; px[u] = nullptr; pt[u] = nullptr; sidx[u] = 0; rr[u] = 0;
            if (g < a.total_rows) {
                int s = 0;
#pragma unroll
                for (int k = 1; k < YB_MAX_SCALES; ++k)
                    if (k < a.S && g >= a.sc[k].row_begin) s = k;
                const uint32_t r = g - a.sc[s].row_begin;
                px[u] = reinterpret_cast<const float*>(a.sc[s].pred) + (size_t)r * a.row;
                pt[u] = a.sc[s].tgt + (size_t)r * a.row;
                xo[u] = __ldg(px[u] + 4);
                to[u] = __ldg(pt[u] + 4);
                sidx[u] = s; rr[u] = r;
            }
        }
#pragma unroll
        for (int u = 0; u < kEvalIlp; ++u) {
            if (!px[u]) continue;
            // .item() -> python float: the threshold tests run in double (:1003-1006)
            const bool p_on = (double)sigmoidf_ref(xo[u]) > a.conf;
            const bool t_on = (double)to[u] > a.conf;
            if (p_on && t_on) {
                const EvalScale& L = a.sc[sidx[u]];
                uint32_t b, gy, gx, an;
                head_row_coords(L, rr[u], b, gy, gx, an);
                const float aw = __ldg(L.anchors + an * 2), ah = __ldg(L.anchors + an * 2 + 1);
                const float pb[4] = {box_xy(sigmoidf_ref(__ldg(px[u])), (float)gx, L.inv_w),
                                     box_xy(sigmoidf_ref(__ldg(px[u] + 1)), (float)gy, L.inv_h),
                                     box_wh(sigmoidf_ref(__ldg(px[u] + 2)), aw, a.inv_img),
                                     box_wh(sigmoidf_ref(__ldg(px[u] + 3)), ah, a.inv_img)};
                const float tb[4] = {__ldg(pt[u]), __ldg(pt[u] + 1), __ldg(pt[u] + 2), __ldg(pt[u] + 3)};
                if (box_iou_xywh(pb, tb) > a.iou_thr) ++tp;  // :1012 fp32 tensor > python scalar
                else ++fp;
            } else if (p_on) {
                ++fp;  // :1016-1018
            } else if (t_on) {
                ++fn;  // :1019-1021
            }
        }
    }
    tp = __reduce_add_sync(0xffffffffu, tp);
    fp = __reduce_add_sync(0xffffffffu, fp);
    fn = __reduce_add_sync(0xffffffffu, fn);
    if ((threadIdx.x & 31) == 0) {
        if (tp) atomicAdd(&s_cnt[0], tp);
        if (fp) atomicAdd(&s_cnt[1], fp);
        if (fn) atomicAdd(&s_cnt[2], fn);
    }
    __syncthreads();
    if (threadIdx.x < 3 && s_cnt[threadIdx.x]) atomicAdd(a.counts + threadIdx.x, (unsigned long long)s_cnt[threadIdx.x]);
}

}  // namespace yb

extern "C" int yb_eval_counts(const yb_heads_desc* d, const float* const* targets_host, double conf_threshold,
                              double iou_threshold, long long* counts3, void* stream) {
    using namespace yb;
    YB_CHECK_ARG(d && targets_host && counts3, "eval_counts: null argument");
    int rc = heads_check(*d, "eval_counts", 0, false, false, true);
    if (rc) return rc;
    if (d->B == 0) return 0;
    EvalArgs a;
    a.S = d->S; a.A = d->A; a.row = 5 + d->nc;
    a.inv_img = 1.0f / d->img_size;
    a.iou_thr = (float)iou_threshold;
    a.conf = conf_threshold;
    a.counts = reinterpret_cast<unsigned long long*>(counts3);
    unsigned long long total = 0;
    for (int s = 0; s < d->S; ++s) {
        YB_CHECK_ARG(targets_host[s], "eval_counts: null targets at scale %d", s);
        EvalScale& L = a.sc[s];
        head_scale_fill(L, *d, s);
        L.tgt = targets_host[s];
        L.row_begin = (uint32_t)total;
        total += (unsigned long long)L.img_rows * d->B;
    }
    // the ILP-4 walk's row index g0 + 3 * stride must not wrap
    YB_CHECK_ARG(total < (1ull << 32) - (1ull << 24), "eval_counts: too many rows");
    a.total_rows = (uint32_t)total;
    const unsigned long long per_cta = (unsigned long long)kEvalThreads * kEvalIlp;
    unsigned long long want = (total + per_cta - 1) / per_cta;
    const unsigned long long cap = (unsigned long long)sm_count() * 8;
    const int blocks = (int)(want < cap ? (want ? want : 1) : cap);
    cudaStream_t st = (cudaStream_t)stream;
    YB_LAUNCH("eval_count_kernel", st, eval_count_kernel<<<blocks, kEvalThreads, 0, st>>>(a));
    return 0;
}
