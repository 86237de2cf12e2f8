// yb_map.cu — COCO-style mAP (COCOeval.evaluateImg + accumulate, bbox, area "all", no crowd) on the device.
//
// Stage 1, map_match_kernel: one CTA per image.  The image's ground truths are staged in shared memory as fp64
// corners; warp t runs COCO's greedy matching for IoU threshold t over the kept detections in keep order (its
// lanes cover the ground truths, a warp arg-max resolves each step), so the T thresholds proceed side by side.
// Output: one 12-byte record (score, class, TP bit per threshold) per detection slot, plus the per-class
// ground-truth counts.  Stage 2, map_precision_kernel: one CTA per class over the records the caller sorted by
// (class, descending score, image order); a block scan of the T TP counts writes the precision at every TP
// position, then the suffix maximum gives the (T,R,nc) precision table and the (T,nc) recall table.
// Every fp64 expression is the oracle's (oracle/map_ref.py) operation for operation (-fmad=false).
#include "yb_common.cuh"
#include "yb_iou.cuh"

namespace yb {

constexpr int kPrecThreads = 256;

struct MatchArgs {
    const float4* boxes;
    const float* scores;
    const int64_t* classes;
    const int64_t* keep;
    const int* n_keep;
    const double* labels;
    const int* n_gt;
    const double* letterbox;
    const double* thr;
    yb_map_record* records;
    unsigned long long* gt_count;
    int* status;
    int cap, slots, max_gt, nc, T;
};

__global__ void __launch_bounds__(512) map_match_kernel(const MatchArgs a) {
    extern __shared__ __align__(16) unsigned char smem[];
    const int chunk = blockDim.x;
    const int words = (a.max_gt + 31) / 32;
    GtBox* s_gt = reinterpret_cast<GtBox*>(smem);
    float4* s_box = reinterpret_cast<float4*>(s_gt + a.max_gt);
    int* s_gcls = reinterpret_cast<int*>(s_box + chunk);
    int* s_dcls = s_gcls + a.max_gt;
    float* s_score = reinterpret_cast<float*>(s_dcls + chunk);
    unsigned int* s_tp = reinterpret_cast<unsigned int*>(s_score + chunk);
    unsigned int* s_matched = s_tp + chunk;   // [T][words]: ground truth g already taken at threshold t

    const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int nk = a.n_keep[b];
    int bad = 0;
    if (nk < 0) bad |= 2;
    const int nd = nk < 0 ? 0 : min(nk, a.slots);
    const int ng = min(max(a.n_gt[b], 0), a.max_gt);
    const double ow = a.letterbox[(size_t)b * 5 + 0], oh = a.letterbox[(size_t)b * 5 + 1];
    for (int g = tid; g < ng; g += blockDim.x) {
        const double* L = a.labels + ((size_t)b * a.max_gt + g) * 5;
        const double xc = L[1], yc = L[2], w = L[3], h = L[4];
        s_gt[g] = GtBox{(xc - w / 2.0) * ow, (yc - h / 2.0) * oh, (xc + w / 2.0) * ow, (yc + h / 2.0) * oh};
        int c = 0;
        if (a.nc > 1) {   // nc == 1: every ground truth is class 0 (train.py:201-202)
            c = (int)L[0];
            if (c < 0 || c >= a.nc) { bad |= 1; c = -1; }
        }
        s_gcls[g] = c;
        if (c >= 0) atomicAdd(a.gt_count + c, 1ull);
    }
    for (int i = tid; i < a.T * words; i += blockDim.x) s_matched[i] = 0u;

    yb_map_record* rec = a.records + (size_t)b * a.slots;
    for (int j0 = 0; j0 < nd; j0 += chunk) {
        const int j = j0 + tid;
        __syncthreads();   // previous chunk consumed; on the first pass: ground truths staged
        if (j < nd) {
            const size_t src = (size_t)b * a.cap + (size_t)a.keep[(size_t)b * a.cap + j];
            const int64_t c = a.classes[src];
            s_box[tid] = a.boxes[src];
            s_score[tid] = a.scores[src];
            s_dcls[tid] = (c >= 0 && c < a.nc) ? (int)c : -1;
            if (!(c >= 0 && c < a.nc)) bad |= 1;
            s_tp[tid] = 0u;
        }
        __syncthreads();
        if (warp < a.T) {
            const double thr = a.thr[warp];
            unsigned int* matched = s_matched + warp * words;
            const int n = min(chunk, nd - j0);
            for (int k = 0; k < n; ++k) {
                const int c = s_dcls[k];
                if (c < 0) continue;
                const float4 q = s_box[k];
                const GtBox d{(double)q.x, (double)q.y, (double)q.z, (double)q.w};
                double best = -INFINITY;
                int bi = -1;
                for (int g = lane; g < ng; g += 32) {
                    if (s_gcls[g] != c || ((matched[g >> 5] >> lane) & 1u)) continue;
                    const double iou = corner_iou(d, s_gt[g]);
                    if (iou >= thr && iou >= best) { best = iou; bi = g; }   // later ground truth wins ties
                }
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) {
                    const double ob = __shfl_xor_sync(0xffffffffu, best, o);
                    const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
                    if (oi >= 0 && (bi < 0 || ob > best || (ob == best && oi > bi))) { best = ob; bi = oi; }
                }
                if (bi >= 0 && lane == 0) {
                    matched[bi >> 5] |= 1u << (bi & 31);
                    atomicOr(s_tp + k, 1u << warp);
                }
                __syncwarp();
            }
        }
        __syncthreads();
        if (j < nd) rec[j] = yb_map_record{s_score[tid], s_dcls[tid], (uint16_t)s_tp[tid], 0};
    }
    for (int j = nd + tid; j < a.slots; j += blockDim.x) rec[j] = yb_map_record{0.0f, -1, 0, 0};
    if (bad) atomicOr(a.status, bad);
}

// The first record of every class c >= 0 is seg[c]; seg[nc] ends the last one (records of class -1 follow).
struct PrecArgs {
    const yb_map_record* rec;
    const long long* seg;
    const unsigned long long* gt_count;
    const double* rec_thr;
    double* ws;
    long long ws_elems;
    double* precision;   // (T,R,nc)
    double* recall;      // (T,nc)
    int* status;
    int nc, T, R;
};

__global__ void __launch_bounds__(kPrecThreads) map_precision_kernel(const PrecArgs a) {
    constexpr int kWarps = kPrecThreads / 32;
    __shared__ unsigned int s_wcnt[kWarps][YB_MAP_MAX_T];
    __shared__ long long s_carry[YB_MAP_MAX_T];
    __shared__ double s_wmax[kWarps];
    __shared__ double s_env_carry;
    __shared__ long long s_base;
    const int c = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const long long s0 = a.seg[c], nd = a.seg[c + 1] - s0;
    const long long ngt = (long long)a.gt_count[c];
    if (tid < YB_MAP_MAX_T) s_carry[tid] = 0;
    if (tid == 0) {
        // this class's rows of the workspace: T rows of min(n_gt, n_det) precisions (k TPs need k <= both)
        long long base = 0;
        for (int i = 0; i < c; ++i) base += min((long long)a.gt_count[i], a.seg[i + 1] - a.seg[i]);
        s_base = base * a.T;
    }
    __syncthreads();
    if (ngt == 0) {   // COCO leaves -1 in both tables for a class without ground truth
        for (int i = tid; i < a.T * a.R; i += kPrecThreads) a.precision[(size_t)i * a.nc + c] = -1.0;
        for (int t = tid; t < a.T; t += kPrecThreads) a.recall[(size_t)t * a.nc + c] = -1.0;
        return;
    }
    const long long rows = min(ngt, nd);
    double* ws = a.ws + s_base;
    if (s_base + rows * a.T > a.ws_elems) {
        if (tid == 0) atomicOr(a.status, 4);
        return;
    }
    // pass 1: cumulative TP/FP counts along the sorted records; the precision at the k-th TP goes to ws[t][k-1]
    const unsigned int lt = (1u << lane) - 1u;
    for (long long i0 = 0; i0 < nd; i0 += kPrecThreads) {
        const long long i = i0 + tid;
        const unsigned int m = i < nd ? a.rec[s0 + i].tp : 0u;
        for (int t = 0; t < a.T; ++t) {
            const unsigned int bal = __ballot_sync(0xffffffffu, (m >> t) & 1u);
            if (lane == 0) s_wcnt[warp][t] = __popc(bal);
        }
        __syncthreads();
        for (int t = 0; t < a.T; ++t) {
            const unsigned int bal = __ballot_sync(0xffffffffu, (m >> t) & 1u);
            if (!((m >> t) & 1u)) continue;
            long long k = s_carry[t] + __popc(bal & lt) + 1;   // TPs up to and including record i
            for (int w = 0; w < warp; ++w) k += s_wcnt[w][t];
            if (k > rows) { atomicOr(a.status, 4); continue; }   // more TPs than ground truths: inconsistent input
            const double tp = (double)k, fp = (double)(i + 1 - k);
            ws[t * rows + k - 1] = tp / (fp + tp + 2.220446049250313e-16);   // COCO: tp / (fp + tp + np.spacing(1))
        }
        __syncthreads();
        if (tid < a.T) {
            long long s = 0;
            for (int w = 0; w < kWarps; ++w) s += s_wcnt[w][tid];
            s_carry[tid] += s;
        }
        __syncthreads();
    }
    for (int t = tid; t < a.T; t += kPrecThreads)
        a.recall[(size_t)t * a.nc + c] = nd > 0 ? (double)s_carry[t] / (double)ngt : 0.0;
    // pass 2: suffix maximum of each row (COCO's precision envelope, restricted to TP positions)
    for (int t = 0; t < a.T; ++t) {
        const long long K = min(s_carry[t], rows);
        double* row = ws + t * rows;
        if (tid == 0) s_env_carry = 0.0;
        for (long long hi = K; hi > 0; hi -= kPrecThreads) {
            const long long idx = hi - kPrecThreads + tid;
            double v = idx >= 0 ? row[idx] : 0.0;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const double u = __shfl_down_sync(0xffffffffu, v, o);
                if (lane + o < 32) v = fmax(v, u);
            }
            if (lane == 0) s_wmax[warp] = v;
            __syncthreads();
            double after = s_env_carry;
            for (int w = warp + 1; w < kWarps; ++w) after = fmax(after, s_wmax[w]);
            if (idx >= 0) row[idx] = fmax(v, after);
            __syncthreads();
            if (tid == 0) {
                double m = s_env_carry;
                for (int w = 0; w < kWarps; ++w) m = fmax(m, s_wmax[w]);
                s_env_carry = m;
            }
            __syncthreads();
        }
    }
    __syncthreads();
    // pass 3: precision at recall r = envelope at the first TP count k with k / n_gt >= r, 0 if there is none
    for (int i = tid; i < a.T * a.R; i += kPrecThreads) {
        const int t = i / a.R, r = i - t * a.R;
        const long long K = min(s_carry[t], rows);
        const double rt = a.rec_thr[r], n = (double)ngt;
        long long k = 1;
        if (rt > 0.0) {
            const double e = ceil(rt * n);
            k = e > n + 1.0 ? ngt + 1 : (e < 1.0 ? 1 : (long long)e);
            while (k > 1 && (double)(k - 1) / n >= rt) --k;
            while (k <= ngt && !((double)k / n >= rt)) ++k;
        }
        a.precision[(size_t)i * a.nc + c] = k <= K ? ws[t * rows + k - 1] : 0.0;
    }
}

}  // namespace yb

extern "C" int yb_map_match(const float* boxes, const float* scores, const int64_t* classes, const int64_t* keep,
                            const int* n_keep, int B, int cap, int max_det, const double* labels, const int* n_gt,
                            const double* letterbox, int max_gt, int nc, const double* iou_thr, int T,
                            yb_map_record* records, long long* gt_count, int* status, void* stream) {
    using namespace yb;
    YB_CHECK_ARG(B >= 0 && cap >= 0 && max_det >= 0 && nc >= 1, "map_match: bad B/cap/max_det/nc");
    YB_CHECK_ARG(T >= 1 && T <= YB_MAP_MAX_T, "map_match: 1 <= T <= %d thresholds", YB_MAP_MAX_T);
    YB_CHECK_ARG(max_gt >= 0 && max_gt <= YB_MAP_MAX_GT, "map_match: max_gt must be in [0, %d]", YB_MAP_MAX_GT);
    if (B == 0) return 0;
    const int slots = max_det < cap ? max_det : cap;
    YB_CHECK_ARG(n_keep && n_gt && letterbox && iou_thr && gt_count && status && (slots == 0 || records),
                 "map_match: null pointer");
    YB_CHECK_ARG(cap == 0 || (boxes && scores && classes && keep && aligned16(boxes)), "map_match: null or unaligned candidates");
    YB_CHECK_ARG(max_gt == 0 || labels, "map_match: null labels");
    MatchArgs a{reinterpret_cast<const float4*>(boxes), scores, classes, keep, n_keep, labels, n_gt, letterbox, iou_thr,
                records, reinterpret_cast<unsigned long long*>(gt_count), status, cap, slots, max_gt, nc, T};
    const int threads = T * 32 < 128 ? 128 : T * 32;
    const size_t smem = (size_t)max_gt * (sizeof(GtBox) + sizeof(int)) + (size_t)threads * (sizeof(float4) + 3 * sizeof(int)) +
                        (size_t)T * ((max_gt + 31) / 32) * sizeof(unsigned int);
    if (smem > 48 * 1024) YB_CUDA(cudaFuncSetAttribute(map_match_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    cudaStream_t st = (cudaStream_t)stream;
    YB_LAUNCH("map_match_kernel", st, map_match_kernel<<<B, threads, smem, st>>>(a));
    return 0;
}

extern "C" size_t yb_map_workspace_bytes(long long n_records, long long n_gt_total, int T) {
    if (n_records < 0 || n_gt_total < 0 || T < 1) return 0;
    const long long rows = n_records < n_gt_total ? n_records : n_gt_total;
    return (size_t)(rows > 0 ? rows : 1) * (size_t)T * sizeof(double);
}

extern "C" int yb_map_precision(const yb_map_record* records, const long long* seg, const long long* gt_count, int nc,
                                int T, const double* recall_thr, int R, double* precision, double* recall, void* ws,
                                size_t ws_bytes, int* status, void* stream) {
    using namespace yb;
    YB_CHECK_ARG(nc >= 1 && T >= 1 && T <= YB_MAP_MAX_T && R >= 1, "map_precision: bad nc/T/R");
    YB_CHECK_ARG(seg && gt_count && recall_thr && precision && recall && ws && status, "map_precision: null pointer");
    YB_CHECK_ARG(nc <= 2147483647 / (T * R), "map_precision: table too large");
    PrecArgs a{records, seg, reinterpret_cast<const unsigned long long*>(gt_count), recall_thr, (double*)ws,
               (long long)(ws_bytes / sizeof(double)), precision, recall, status, nc, T, R};
    cudaStream_t st = (cudaStream_t)stream;
    YB_LAUNCH("map_precision_kernel", st, map_precision_kernel<<<nc, kPrecThreads, 0, st>>>(a));
    return 0;
}
