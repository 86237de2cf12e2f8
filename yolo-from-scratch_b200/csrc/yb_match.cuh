// yb_match.cuh — the per-image front end shared by the mAP (yb_map.cu), COCO (yb_coco.cu) and validation report
// (yb_report.cu) match kernels: their common inputs, the fp64 ground-truth staging, the kept-detection load, the
// corner IoU, COCO's greedy matching step and the host-side checks of the shared arguments.
#pragma once
#include "yb_common.cuh"

namespace yb {

// the current device's opt-in shared memory per block (48 KB if it cannot be read)
static inline int max_smem_optin() {
    int dev = 0, v = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&v, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev) != cudaSuccess)
        return 48 * 1024;
    return v;
}

// The per-batch inputs every match kernel takes (include/yolo_b200.h, yb_map_match).  slots = min(max_det, cap).
struct MatchInputs {
    const float4* boxes;
    const float* scores;
    const int64_t* classes;
    const int64_t* keep;
    const int* n_keep;
    const double* labels;
    const int* n_gt;
    const double* letterbox;
    int cap, slots, max_gt, nc;
};

struct GtBox {
    double x1, y1, x2, y2;
};

// compute_iou_corners (train.py:1064-1084): 0 when the union is not positive
__device__ __forceinline__ double corner_iou(const GtBox& a, const GtBox& b) {
    const double iw = fmax(0.0, fmin(a.x2, b.x2) - fmax(a.x1, b.x1));
    const double ih = fmax(0.0, fmin(a.y2, b.y2) - fmax(a.y1, b.y1));
    const double inter = iw * ih;
    const double uni = (a.x2 - a.x1) * (a.y2 - a.y1) + (b.x2 - b.x1) * (b.y2 - b.y1) - inter;
    return uni > 0.0 ? inter / uni : 0.0;
}

// Image b of a batch: its kept detections (at most slots; none when NMS failed, which sets YB_MAP_NMS_FAILED in
// bad), its ground truths (at most max_gt) and the original image size the labels are normalised to.
struct MatchImage {
    int b, nd, ng;
    double ow, oh;
};

__device__ __forceinline__ MatchImage match_image(const MatchInputs& in, int b, int& bad) {
    const int nk = in.n_keep[b];
    bad = nk < 0 ? YB_MAP_NMS_FAILED : 0;
    return MatchImage{b, nk < 0 ? 0 : min(nk, in.slots), min(max(in.n_gt[b], 0), in.max_gt),
                      in.letterbox[(size_t)b * 5 + 0], in.letterbox[(size_t)b * 5 + 1]};
}

// Ground truth g of the image as fp64 corners in original-image pixels; returns its class, -1 (and
// YB_MAP_BAD_CLASS in bad) when it is outside [0, nc).
__device__ __forceinline__ int stage_gt(const MatchInputs& in, const MatchImage& im, int g, GtBox& box, int& bad) {
    const double* L = in.labels + ((size_t)im.b * in.max_gt + g) * 5;
    const double xc = L[1], yc = L[2], w = L[3], h = L[4];
    box = GtBox{(xc - w / 2.0) * im.ow, (yc - h / 2.0) * im.oh, (xc + w / 2.0) * im.ow, (yc + h / 2.0) * im.oh};
    int c = 0;
    if (in.nc > 1) {   // nc == 1: every ground truth is class 0 (train.py:201-202)
        c = (int)L[0];
        if (c < 0 || c >= in.nc) { bad |= YB_MAP_BAD_CLASS; c = -1; }
    }
    return c;
}

// The j-th kept detection of the image: its index into the candidate arrays, and its class, -1 (and
// YB_MAP_BAD_CLASS in bad) when it is outside [0, nc).
struct Kept {
    size_t src;
    int cls;
};

__device__ __forceinline__ Kept load_kept(const MatchInputs& in, const MatchImage& im, int j, int& bad) {
    const size_t src = (size_t)im.b * in.cap + (size_t)in.keep[(size_t)im.b * in.cap + j];
    const int64_t c = in.classes[src];
    const bool ok = c >= 0 && c < in.nc;
    if (!ok) bad |= YB_MAP_BAD_CLASS;
    return Kept{src, ok ? (int)c : -1};
}

// COCO's greedy matching (evaluateImg) at IoU threshold thr, run by one warp over the n staged detections in keep
// order.  Each detection of a class >= 0 takes, among the not yet matched ground truths of its class with IoU >= thr
// (a NaN IoU never matches), the largest by (not ignored, IoU, index): the later ground truth wins ties.  It then sets
// bit `bit` of its s_tp entry, or of its s_ig entry when that ground truth is ignored.  The lanes scan g = lane,
// lane + 32, ... and a warp arg-max resolves each step.  Without kIgnore every ground truth counts as not ignored, and
// s_gnig and s_ig are not read.  matched[words]: ground truth g already taken at this threshold.
template <bool kIgnore>
__device__ __forceinline__ void greedy_match(int n, const float4* s_box, const int* s_dcls, int ng, const GtBox* s_gt,
                                             const int* s_gcls, const int* s_gnig, double thr, int bit,
                                             unsigned int* matched, unsigned int* s_tp, unsigned int* s_ig) {
    const int lane = threadIdx.x & 31;
    for (int k = 0; k < n; ++k) {
        const int c = s_dcls[k];
        if (c < 0) continue;
        const float4 q = s_box[k];
        const GtBox d{(double)q.x, (double)q.y, (double)q.z, (double)q.w};
        double best = -INFINITY;
        int bn = kIgnore ? 0 : 1, bi = -1;   // bn: the best one is not ignored
        for (int g = lane; g < ng; g += 32) {
            if (s_gcls[g] != c || ((matched[g >> 5] >> lane) & 1u)) continue;
            const double iou = corner_iou(d, s_gt[g]);
            if (!(iou >= thr)) continue;
            const int nig = kIgnore ? s_gnig[g] : 1;
            if (nig > bn || (nig == bn && iou >= best)) { best = iou; bn = nig; bi = g; }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const double ob = __shfl_xor_sync(0xffffffffu, best, o);
            const int on = kIgnore ? __shfl_xor_sync(0xffffffffu, bn, o) : 1;
            const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
            if (oi >= 0 && (bi < 0 || on > bn || (on == bn && (ob > best || (ob == best && oi > bi))))) {
                best = ob; bn = on; bi = oi;
            }
        }
        if (bi >= 0 && lane == 0) {
            matched[bi >> 5] |= 1u << (bi & 31);
            atomicOr((bn ? s_tp : s_ig) + k, 1u << bit);
        }
        __syncwarp();
    }
}

// The checks of the arguments every match entry point takes, with `who` prefixing each message, then the opt-in to
// smem bytes of dynamic shared memory for `kernel`.  B == 0 needs no pointer and no launch; own_ptrs: the caller's
// own pointers are all set.
template <typename Kernel>
static inline int check_match(const char* who, Kernel* kernel, const MatchInputs& in, int B, int max_det,
                              bool own_ptrs, size_t smem) {
    YB_CHECK_ARG(B >= 0 && in.cap >= 0 && max_det >= 0 && in.nc >= 1, "%s: bad B/cap/max_det/nc", who);
    YB_CHECK_ARG(in.max_gt >= 0 && in.max_gt <= YB_MAP_MAX_GT, "%s: max_gt must be in [0, %d]", who, YB_MAP_MAX_GT);
    if (B == 0) return 0;
    YB_CHECK_ARG(in.n_keep && in.n_gt && in.letterbox && own_ptrs, "%s: null pointer", who);
    YB_CHECK_ARG(in.cap == 0 || (in.boxes && in.scores && in.classes && in.keep && aligned16(in.boxes)),
                 "%s: null or unaligned candidates", who);
    YB_CHECK_ARG(in.max_gt == 0 || in.labels, "%s: null labels", who);
    YB_CHECK_ARG(smem <= (size_t)max_smem_optin(),
                 "%s: %zu bytes of shared memory (max_gt = %d, min(max_det, cap) = %d, nc = %d) exceed one CTA", who,
                 smem, in.max_gt, in.slots, in.nc);
    if (smem > 48 * 1024) YB_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    return 0;
}

}  // namespace yb
