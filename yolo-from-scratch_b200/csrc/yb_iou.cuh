// yb_iou.cuh — the fp64 ground-truth box and corner IoU shared by the mAP (yb_map.cu), COCO (yb_coco.cu) and
// validation report (yb_report.cu) kernels, and the shared-memory limit their hosts check the staging against.
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

}  // namespace yb
