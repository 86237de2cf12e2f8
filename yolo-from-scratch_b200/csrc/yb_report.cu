// yb_report.cu — the validation report's per-image statistics on the device: the confusion matrix (rows predicted
// class, columns true class, index nc background), the images per class and the confidence histograms of the
// precision / recall / F1 curves; the header states the semantics.
//
// report_match_kernel: one CTA per image, enqueued after yb_map_match on the same batch.  The image's ground truths
// are staged in shared memory as fp64 corners (map_match_kernel's conversion).  The matrix's two-step unique
// matching is class-agnostic:
//   step 1: each detection d above cm_conf (one thread each) scans every ground truth and picks the one with the
//           largest IoU > cm_iou, the lower index on equal IoU; it records (g, IoU) and atomicMax-es the IoU's
//           bits + 1 into g's slot (a non-negative double's bits order like an integer; 0 marks "not picked");
//   step 2: the detections whose IoU equals g's maximum atomicMin their keep position into g's slot, so g keeps
//           the earliest of them.
// The histograms bin every record of the image by its score: bin j holds the scores in (grid[j], grid[j+1]], so a
// suffix sum counts the scores above grid[k] without a sort.  Every global count goes through a warp-aggregated
// atomicAdd (__match_any_sync on the destination: one atomic per distinct cell per warp), which keeps the nc = 1
// case, where a whole batch lands on four matrix cells and a few bins, from serialising on single addresses.
#include <climits>
#include "yb_common.cuh"
#include "yb_iou.cuh"

namespace yb {

constexpr int kReportThreads = 256;

struct ReportArgs {
    const float4* boxes;
    const float* scores;
    const int64_t* classes;
    const int64_t* keep;
    const int* n_keep;
    const double* labels;
    const int* n_gt;
    const double* letterbox;
    const yb_map_record* records;
    const double* grid;
    unsigned long long* confusion;   // (nc+1, nc+1)
    unsigned long long* images;      // (nc)
    unsigned long long* det_hist;    // (nc, K)
    unsigned long long* tp_hist;     // (nc, K)
    int* status;
    double cm_conf, cm_iou;
    int cap, slots, max_gt, nc, K, t_curve;
};

// Every lane of the warp calls this.  The lanes with on set and equal idx add, through their lowest lane, the number
// of them whose bit is set in sub to dst[idx].
__device__ __forceinline__ void warp_add(unsigned long long* dst, unsigned long long idx, bool on, unsigned int sub) {
    const unsigned int peers = __match_any_sync(0xffffffffu, on ? idx : ~0ull);
    const unsigned int n = __popc(peers & sub);
    if (on && n && (int)(threadIdx.x & 31) == __ffs(peers) - 1) atomicAdd(dst + idx, (unsigned long long)n);
}

__global__ void __launch_bounds__(kReportThreads) report_match_kernel(const ReportArgs a) {
    extern __shared__ __align__(16) unsigned char smem[];
    GtBox* s_gt = reinterpret_cast<GtBox*>(smem);
    unsigned long long* s_key = reinterpret_cast<unsigned long long*>(s_gt + a.max_gt);   // [max_gt] best IoU bits + 1
    unsigned long long* s_dkey = s_key + a.max_gt;                                        // [slots] d's IoU bits + 1
    int* s_gcls = reinterpret_cast<int*>(s_dkey + a.slots);                               // [max_gt] -1: not in G
    int* s_pos = s_gcls + a.max_gt;                                                       // [max_gt] keep position g keeps
    int* s_pick = s_pos + a.max_gt;                                                       // [slots] -2: not in D, -1: none
    int* s_dcls = s_pick + a.slots;                                                       // [slots]
    int* s_seen = s_dcls + a.slots;                                                       // [nc]

    const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31;
    const int nk = a.n_keep[b];
    int bad = nk < 0 ? YB_MAP_NMS_FAILED : 0;
    const int nd = nk < 0 ? 0 : min(nk, a.slots);
    const int ng = min(max(a.n_gt[b], 0), a.max_gt);
    const double ow = a.letterbox[(size_t)b * 5 + 0], oh = a.letterbox[(size_t)b * 5 + 1];
    for (int c = tid; c < a.nc; c += blockDim.x) s_seen[c] = 0;
    __syncthreads();
    for (int g = tid; g < ng; g += blockDim.x) {
        const double* L = a.labels + ((size_t)b * a.max_gt + g) * 5;
        const double xc = L[1], yc = L[2], w = L[3], h = L[4];
        s_gt[g] = GtBox{(xc - w / 2.0) * ow, (yc - h / 2.0) * oh, (xc + w / 2.0) * ow, (yc + h / 2.0) * oh};
        int c = 0;
        if (a.nc > 1) {   // nc == 1: every ground truth is class 0 (train.py:201-202)
            c = (int)L[0];
            if (c < 0 || c >= a.nc) { bad |= YB_MAP_BAD_CLASS; c = -1; }
        }
        s_gcls[g] = c;
        s_key[g] = 0ull;
        s_pos[g] = INT_MAX;
        if (c >= 0 && atomicExch(s_seen + c, 1) == 0) atomicAdd(a.images + c, 1ull);
    }
    __syncthreads();
    // step 1: each d in D picks its ground truth
    for (int j = tid; j < nd; j += blockDim.x) {
        const size_t src = (size_t)b * a.cap + (size_t)a.keep[(size_t)b * a.cap + j];
        const int64_t c = a.classes[src];
        int pick = -2;
        unsigned long long key = 0ull;
        if (!(c >= 0 && c < a.nc)) {
            bad |= YB_MAP_BAD_CLASS;
        } else if ((double)a.scores[src] > a.cm_conf) {   // a NaN score never passes
            const float4 q = a.boxes[src];
            const GtBox d{(double)q.x, (double)q.y, (double)q.z, (double)q.w};
            double best = 0.0;
            pick = -1;
            for (int g = 0; g < ng; ++g) {
                if (s_gcls[g] < 0) continue;
                const double iou = corner_iou(d, s_gt[g]);
                if (iou > a.cm_iou && (pick < 0 || iou > best)) { best = iou; pick = g; }   // a NaN IoU never matches
            }
            if (pick >= 0) {
                key = (unsigned long long)__double_as_longlong(best) + 1ull;
                atomicMax(s_key + pick, key);
            }
        }
        s_pick[j] = pick;
        s_dkey[j] = key;
        s_dcls[j] = (int)c;
    }
    __syncthreads();
    // step 2: each picked g keeps the earliest of the detections at its largest IoU
    for (int j = tid; j < nd; j += blockDim.x) {
        const int g = s_pick[j];
        if (g >= 0 && s_dkey[j] == s_key[g]) atomicMin(s_pos + g, j);
    }
    __syncthreads();
    const unsigned long long side = (unsigned long long)a.nc + 1;
    for (int j0 = tid - lane; j0 < nd; j0 += blockDim.x) {   // whole warps: warp_add needs every lane
        const int j = j0 + lane;
        const int g = j < nd ? s_pick[j] : -2;
        unsigned long long cell = 0ull;
        if (g >= -1) cell = (unsigned long long)s_dcls[j] * side + (unsigned long long)(g >= 0 && s_pos[g] == j ? s_gcls[g] : a.nc);
        warp_add(a.confusion, cell, g >= -1, 0xffffffffu);
    }
    for (int g0 = tid - lane; g0 < ng; g0 += blockDim.x) {   // ground truths no detection picked: background row
        const int g = g0 + lane;
        const bool on = g < ng && s_gcls[g] >= 0 && s_key[g] == 0ull;
        warp_add(a.confusion, on ? (unsigned long long)a.nc * side + (unsigned long long)s_gcls[g] : 0ull, on, 0xffffffffu);
    }
    // histograms: bin j = #{k : grid[k] < score} - 1 of every record with a class and a non-NaN score
    const yb_map_record* rec = a.records + (size_t)b * a.slots;
    for (int j0 = tid - lane; j0 < a.slots; j0 += blockDim.x) {
        const int j = j0 + lane;
        bool on = false, tp = false;
        unsigned long long bin = 0ull;
        if (j < a.slots) {
            const yb_map_record r = rec[j];
            const double s = (double)r.score;
            if (r.cls >= 0 && r.cls < a.nc && s == s) {
                int lo = 0, hi = a.K;
                while (lo < hi) {
                    const int mid = (lo + hi) >> 1;
                    if (__ldg(a.grid + mid) < s) lo = mid + 1; else hi = mid;
                }
                if (lo > 0) {
                    on = true;
                    bin = (unsigned long long)r.cls * (unsigned long long)a.K + (unsigned long long)(lo - 1);
                    tp = (r.tp >> a.t_curve) & 1u;
                }
            }
        }
        warp_add(a.det_hist, bin, on, 0xffffffffu);
        warp_add(a.tp_hist, bin, on, __ballot_sync(0xffffffffu, tp));
    }
    if (bad) atomicOr(a.status, bad);
}

}  // namespace yb

extern "C" int yb_report_match(const float* boxes, const float* scores, const int64_t* classes, const int64_t* keep,
                               const int* n_keep, int B, int cap, int max_det, const double* labels, const int* n_gt,
                               const double* letterbox, int max_gt, int nc, const yb_map_record* records, int t_curve,
                               const double* grid, int K, double cm_conf, double cm_iou, long long* confusion,
                               long long* images, long long* det_hist, long long* tp_hist, int* status, void* stream) {
    using namespace yb;
    YB_CHECK_ARG(B >= 0 && cap >= 0 && max_det >= 0 && nc >= 1, "report_match: bad B/cap/max_det/nc");
    YB_CHECK_ARG(max_gt >= 0 && max_gt <= YB_MAP_MAX_GT, "report_match: max_gt must be in [0, %d]", YB_MAP_MAX_GT);
    YB_CHECK_ARG(t_curve >= 0 && t_curve < YB_MAP_MAX_T, "report_match: t_curve must be in [0, %d)", YB_MAP_MAX_T);
    YB_CHECK_ARG(K >= 1 && (long long)nc * K <= (1ll << 40), "report_match: bad grid size K = %d", K);
    YB_CHECK_ARG(isfinite(cm_conf) && isfinite(cm_iou), "report_match: cm_conf and cm_iou must be finite");
    if (B == 0) return 0;
    const int slots = max_det < cap ? max_det : cap;
    YB_CHECK_ARG(n_keep && n_gt && letterbox && grid && confusion && images && det_hist && tp_hist && status &&
                 (slots == 0 || records), "report_match: null pointer");
    YB_CHECK_ARG(cap == 0 || (boxes && scores && classes && keep && aligned16(boxes)), "report_match: null or unaligned candidates");
    YB_CHECK_ARG(max_gt == 0 || labels, "report_match: null labels");
    const size_t smem = (size_t)max_gt * (sizeof(GtBox) + sizeof(unsigned long long) + 2 * sizeof(int)) +
                        (size_t)slots * (sizeof(unsigned long long) + 2 * sizeof(int)) + (size_t)nc * sizeof(int);
    YB_CHECK_ARG(smem <= (size_t)max_smem_optin(),
                 "report_match: %zu bytes of shared memory (max_gt = %d, min(max_det, cap) = %d, nc = %d) exceed one CTA",
                 smem, max_gt, slots, nc);
    if (smem > 48 * 1024) YB_CUDA(cudaFuncSetAttribute(report_match_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    ReportArgs a{reinterpret_cast<const float4*>(boxes), scores, classes, keep, n_keep, labels, n_gt, letterbox, records, grid,
                 reinterpret_cast<unsigned long long*>(confusion), reinterpret_cast<unsigned long long*>(images),
                 reinterpret_cast<unsigned long long*>(det_hist), reinterpret_cast<unsigned long long*>(tp_hist), status,
                 cm_conf, cm_iou, cap, slots, max_gt, nc, K, t_curve};
    cudaStream_t st = (cudaStream_t)stream;
    YB_LAUNCH("report_match_kernel", st, report_match_kernel<<<B, kReportThreads, smem, st>>>(a));
    return 0;
}
