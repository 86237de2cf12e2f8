// yb_coco.cu — COCO's bbox summary (COCOeval.evaluateImg + accumulate with area ranges and per-(image, category)
// maxDets, no crowd) on the device; the header states the semantics.
//
// Stage 1, coco_match_kernel: one CTA per (image, area range).  The image's ground truths are staged in shared
// memory as fp64 corners with their "ignored in this range" flag; warp t runs COCO's greedy matching for IoU
// threshold t over the kept detections in keep order, a warp arg-max on (not ignored, IoU, index) resolving each
// step, exactly as map_match_kernel does with the flag as the leading key.  The CTA of range 0 also writes each
// detection's rank within its (image, class): warp 0 groups 32 detections at a time by class with
// __match_any_sync and carries per-class counts in shared memory.  Output: one 32-byte record per detection slot
// (score, class, rank, TP and ignored bits per threshold for every range), plus the non-ignored ground-truth
// counts per range and class.
// Stage 2, coco_precision_kernel: one CTA per (class, range) over the records the caller sorted by (class,
// descending score, image order), the M maxDets filters in the same pass.  A block scan of the TP and non-ignored
// counts gives, at every TP, its precision pr and its recall bucket b(k) = max{r : k / npig >= recall_thr[r]};
// a shared-memory (M,T,R) table keeps the largest pr per bucket (a non-negative double's bits order like an
// integer, so an integer atomicMax is exact), and its suffix maximum over r is COCO's precision table.
// Every fp64 expression is the oracle's (oracle/coco_ref.py) operation for operation (-fmad=false).
#include "yb_common.cuh"
#include "yb_iou.cuh"

namespace yb {

constexpr int kCocoPrecThreads = 256;

struct CocoMatchArgs {
    const float4* boxes;
    const float* scores;
    const int64_t* classes;
    const int64_t* keep;
    const int* n_keep;
    const double* labels;
    const int* n_gt;
    const double* letterbox;
    const double* thr;
    yb_coco_record* records;
    unsigned long long* gt_count;   // (A, nc)
    int* status;
    double rng[2 * YB_COCO_MAX_A];
    int cap, slots, max_gt, nc, T, A;
};

__device__ __forceinline__ bool outside(double area, double lo, double hi) { return area < lo || area > hi; }

__global__ void __launch_bounds__(512) coco_match_kernel(const CocoMatchArgs a) {
    extern __shared__ __align__(16) unsigned char smem[];
    const int chunk = blockDim.x;
    const int words = (a.max_gt + 31) / 32;
    GtBox* s_gt = reinterpret_cast<GtBox*>(smem);
    float4* s_box = reinterpret_cast<float4*>(s_gt + a.max_gt);
    int* s_gcls = reinterpret_cast<int*>(s_box + chunk);
    int* s_gnig = s_gcls + a.max_gt;              // 1: the ground truth is inside this range (not ignored)
    int* s_dcls = s_gnig + a.max_gt;
    int* s_dout = s_dcls + chunk;                 // 1: the detection is outside this range
    int* s_rank = s_dout + chunk;
    float* s_score = reinterpret_cast<float*>(s_rank + chunk);
    unsigned int* s_tp = reinterpret_cast<unsigned int*>(s_score + chunk);
    unsigned int* s_ig = s_tp + chunk;
    unsigned int* s_matched = s_ig + chunk;       // [T][words]: ground truth g already taken at threshold t
    int* s_cnt = reinterpret_cast<int*>(s_matched + a.T * words);   // [nc] detections per class so far (range 0)

    const int b = blockIdx.x, ar = blockIdx.y, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const bool first = ar == 0;   // the CTA of range 0 writes the shared fields and reports the status
    const double lo = a.rng[2 * ar], hi = a.rng[2 * ar + 1];
    const int nk = a.n_keep[b];
    int bad = 0;
    if (nk < 0) bad |= 2;
    const int nd = nk < 0 ? 0 : min(nk, a.slots);
    const int ng = min(max(a.n_gt[b], 0), a.max_gt);
    const double ow = a.letterbox[(size_t)b * 5 + 0], oh = a.letterbox[(size_t)b * 5 + 1];
    for (int g = tid; g < ng; g += blockDim.x) {
        const double* L = a.labels + ((size_t)b * a.max_gt + g) * 5;
        const double xc = L[1], yc = L[2], w = L[3], h = L[4];
        const GtBox box{(xc - w / 2.0) * ow, (yc - h / 2.0) * oh, (xc + w / 2.0) * ow, (yc + h / 2.0) * oh};
        s_gt[g] = box;
        int c = 0;
        if (a.nc > 1) {   // nc == 1: every ground truth is class 0 (train.py:201-202)
            c = (int)L[0];
            if (c < 0 || c >= a.nc) { bad |= 1; c = -1; }
        }
        const int nig = outside((box.x2 - box.x1) * (box.y2 - box.y1), lo, hi) ? 0 : 1;
        s_gcls[g] = c;
        s_gnig[g] = nig;
        if (c >= 0 && nig) atomicAdd(a.gt_count + (size_t)ar * a.nc + c, 1ull);
    }
    for (int i = tid; i < a.T * words; i += blockDim.x) s_matched[i] = 0u;
    if (first)
        for (int i = tid; i < a.nc; i += blockDim.x) s_cnt[i] = 0;

    yb_coco_record* rec = a.records + (size_t)b * a.slots;
    const unsigned int tmask = (1u << a.T) - 1u;
    const double thr_lim = 1.0 - 1e-10;
    for (int j0 = 0; j0 < nd; j0 += chunk) {
        const int j = j0 + tid;
        __syncthreads();   // previous chunk consumed; on the first pass: ground truths and counters staged
        if (j < nd) {
            const size_t src = (size_t)b * a.cap + (size_t)a.keep[(size_t)b * a.cap + j];
            const int64_t c = a.classes[src];
            const float4 q = a.boxes[src];
            s_box[tid] = q;
            s_score[tid] = a.scores[src];
            s_dcls[tid] = (c >= 0 && c < a.nc) ? (int)c : -1;
            if (!(c >= 0 && c < a.nc)) bad |= 1;
            s_dout[tid] = outside(((double)q.z - (double)q.x) * ((double)q.w - (double)q.y), lo, hi) ? 1 : 0;
            s_tp[tid] = 0u;
            s_ig[tid] = 0u;
        }
        __syncthreads();
        const int n = min(chunk, nd - j0);
        if (first && warp == 0) {   // rank within (image, class), 32 detections at a time in keep order
            const unsigned int lt = (1u << lane) - 1u;
            for (int k0 = 0; k0 < n; k0 += 32) {
                const int k = k0 + lane;
                const int c = k < n ? s_dcls[k] : -2;
                const unsigned int peers = __match_any_sync(0xffffffffu, c);
                int base = 0;
                if (c >= 0) base = s_cnt[c];
                __syncwarp();
                if (c >= 0) {
                    const int r = base + __popc(peers & lt);
                    s_rank[k] = r;
                    if ((peers & lt) == 0u) s_cnt[c] = base + __popc(peers);   // the group's first lane
                } else if (k < n) {
                    s_rank[k] = 0;
                }
                __syncwarp();
            }
        }
        if (warp < a.T) {
            const double t0 = a.thr[warp];
            const double thr = thr_lim < t0 ? thr_lim : t0;   // min([t, 1-1e-10])
            unsigned int* matched = s_matched + warp * words;
            for (int k = 0; k < n; ++k) {
                const int c = s_dcls[k];
                if (c < 0) continue;
                const float4 q = s_box[k];
                const GtBox d{(double)q.x, (double)q.y, (double)q.z, (double)q.w};
                double best = -INFINITY;
                int bn = 0, bi = -1;
                for (int g = lane; g < ng; g += 32) {
                    if (s_gcls[g] != c || ((matched[g >> 5] >> lane) & 1u)) continue;
                    const double iou = corner_iou(d, s_gt[g]);
                    if (!(iou >= thr)) continue;   // a NaN IoU never matches
                    const int nig = s_gnig[g];
                    if (nig > bn || (nig == bn && iou >= best)) { best = iou; bn = nig; bi = g; }   // later one wins ties
                }
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) {
                    const double ob = __shfl_xor_sync(0xffffffffu, best, o);
                    const int on = __shfl_xor_sync(0xffffffffu, bn, o);
                    const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
                    if (oi >= 0 && (bi < 0 || on > bn || (on == bn && (ob > best || (ob == best && oi > bi))))) {
                        best = ob; bn = on; bi = oi;
                    }
                }
                if (bi >= 0 && lane == 0) {
                    matched[bi >> 5] |= 1u << (bi & 31);
                    atomicOr((bn ? s_tp : s_ig) + k, 1u << warp);
                }
                __syncwarp();
            }
        }
        __syncthreads();
        if (j < nd) {
            yb_coco_record& r = rec[j];
            const unsigned int tp = s_tp[tid];
            // unmatched detections outside the range are ignored; matched ones keep their state
            const unsigned int ig = s_dout[tid] ? (tmask & ~tp) : s_ig[tid];
            r.tp[ar] = (uint16_t)tp;
            r.ig[ar] = (uint16_t)ig;
            if (first) {
                r.score = s_score[tid];
                r.cls = s_dcls[tid];
                r.rank = (uint16_t)min(s_rank[tid], 65535);
                r.pad = 0;
                for (int q = a.A; q < YB_COCO_MAX_A; ++q) { r.tp[q] = 0; r.ig[q] = 0; }
                r.pad2 = 0u;
            }
        }
    }
    if (first) {
        for (int j = nd + tid; j < a.slots; j += blockDim.x) {
            yb_coco_record& r = rec[j];
            r.score = 0.0f;
            r.cls = -1;
            r.rank = 0;
            r.pad = 0;
            for (int q = 0; q < YB_COCO_MAX_A; ++q) { r.tp[q] = 0; r.ig[q] = 0; }
            r.pad2 = 0u;
        }
        if (bad) atomicOr(a.status, bad);
    }
}

// The first record of class c >= 0 is seg[c]; seg[nc] ends the last one (records of class -1 follow).
struct CocoPrecArgs {
    const yb_coco_record* rec;
    const long long* seg;
    const unsigned long long* gt_count;   // (A, nc)
    const double* rec_thr;
    double* precision;                    // (T,R,nc,A,M)
    double* recall;                       // (T,nc,A,M)
    int* status;
    int max_dets[YB_COCO_MAX_M];
    int nc, A, T, R, M;
};

__global__ void __launch_bounds__(kCocoPrecThreads) coco_precision_kernel(const CocoPrecArgs a) {
    constexpr int kWarps = kCocoPrecThreads / 32;
    extern __shared__ __align__(16) unsigned char smem[];
    unsigned long long* s_best = reinterpret_cast<unsigned long long*>(smem);   // [M][T][R] largest pr per bucket
    double* s_rthr = reinterpret_cast<double*>(s_best + (size_t)a.M * a.T * a.R);
    __shared__ unsigned int s_wtp[YB_COCO_MAX_M][YB_MAP_MAX_T][kWarps];
    __shared__ unsigned int s_wn[YB_COCO_MAX_M][YB_MAP_MAX_T][kWarps];
    __shared__ long long s_ctp[YB_COCO_MAX_M][YB_MAP_MAX_T];   // TPs before the current chunk
    __shared__ long long s_cn[YB_COCO_MAX_M][YB_MAP_MAX_T];    // non-ignored records before the current chunk
    __shared__ int s_md[YB_COCO_MAX_M];
    const int c = blockIdx.x, ar = blockIdx.y, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int MT = a.M * a.T;
    const long long s0 = a.seg[c], nd = a.seg[c + 1] - s0;
    const long long npig = (long long)a.gt_count[(size_t)ar * a.nc + c];
    const size_t cstride = (size_t)a.A * a.M;   // precision / recall: next class
    const size_t pbase = (size_t)c * cstride + (size_t)ar * a.M;
    if (npig == 0) {   // COCO leaves -1 in both tables without (non-ignored) ground truth
        for (int i = tid; i < a.T * a.R * a.M; i += kCocoPrecThreads) {
            const int m = i % a.M, tr = i / a.M;
            a.precision[(size_t)tr * a.nc * cstride + pbase + m] = -1.0;
        }
        for (int i = tid; i < MT; i += kCocoPrecThreads) {
            const int m = i % a.M, t = i / a.M;
            a.recall[(size_t)t * a.nc * cstride + pbase + m] = -1.0;
        }
        return;
    }
    for (int i = tid; i < MT * a.R; i += kCocoPrecThreads) s_best[i] = 0ull;   // +0.0
    for (int r = tid; r < a.R; r += kCocoPrecThreads) s_rthr[r] = a.rec_thr[r];
    if (tid == 0) {
#pragma unroll
        for (int m = 0; m < YB_COCO_MAX_M; ++m) s_md[m] = a.max_dets[m];   // constant indices: no local copy of a
    }
    if (tid < MT) {
        s_ctp[tid / a.T][tid % a.T] = 0;
        s_cn[tid / a.T][tid % a.T] = 0;
    }
    __syncthreads();
    const unsigned int lt = (1u << lane) - 1u;
    const double n_gt = (double)npig;
    for (long long i0 = 0; i0 < nd; i0 += kCocoPrecThreads) {
        const long long i = i0 + tid;
        int rank = 65536;
        unsigned int tpm = 0u, igm = 0u;
        if (i < nd) {
            const yb_coco_record& r = a.rec[s0 + i];
            rank = r.rank;
            tpm = r.tp[ar];
            igm = r.ig[ar];
        }
        for (int m = 0; m < a.M; ++m) {
            const bool counted = rank < s_md[m];
            for (int t = 0; t < a.T; ++t) {
                const unsigned int btp = __ballot_sync(0xffffffffu, counted && ((tpm >> t) & 1u));
                const unsigned int bn = __ballot_sync(0xffffffffu, counted && !((igm >> t) & 1u));
                if (lane == 0) {
                    s_wtp[m][t][warp] = __popc(btp);
                    s_wn[m][t][warp] = __popc(bn);
                }
            }
        }
        __syncthreads();
        for (int m = 0; m < a.M; ++m) {
            const bool counted = rank < s_md[m];
            for (int t = 0; t < a.T; ++t) {
                const bool is_tp = counted && ((tpm >> t) & 1u);
                const unsigned int btp = __ballot_sync(0xffffffffu, is_tp);
                const unsigned int bn = __ballot_sync(0xffffffffu, counted && !((igm >> t) & 1u));
                if (!is_tp) continue;
                long long k = s_ctp[m][t] + __popc(btp & lt) + 1;   // TPs up to and including record i
                long long nn = s_cn[m][t] + __popc(bn & lt) + 1;    // non-ignored records up to and including i
                for (int w = 0; w < warp; ++w) {
                    k += s_wtp[m][t][w];
                    nn += s_wn[m][t][w];
                }
                if (k > npig) { atomicOr(a.status, YB_MAP_INCONSISTENT); continue; }
                const double tp = (double)k, fp = (double)(nn - k);
                const double pr = tp / (fp + tp + 2.220446049250313e-16);   // COCO: tp / (fp + tp + np.spacing(1))
                const double rc = tp / n_gt;
                int lo = 0, hi = a.R;   // number of recall points <= rc
                while (lo < hi) {
                    const int mid = (lo + hi) >> 1;
                    if (s_rthr[mid] <= rc) lo = mid + 1; else hi = mid;
                }
                if (lo > 0)
                    atomicMax(s_best + ((size_t)m * a.T + t) * a.R + (lo - 1), (unsigned long long)__double_as_longlong(pr));
            }
        }
        __syncthreads();
        if (tid < MT) {
            const int m = tid / a.T, t = tid % a.T;
            long long stp = 0, sn = 0;
            for (int w = 0; w < kWarps; ++w) {
                stp += s_wtp[m][t][w];
                sn += s_wn[m][t][w];
            }
            s_ctp[m][t] += stp;
            s_cn[m][t] += sn;
        }
        __syncthreads();
    }
    // recall = rc at the end; precision[r] = suffix maximum of the bucket maxima from r on (0 where there is none)
    for (int i = tid; i < MT; i += kCocoPrecThreads) {
        const int m = i / a.T, t = i % a.T;
        a.recall[(size_t)t * a.nc * cstride + pbase + m] = (double)s_ctp[m][t] / n_gt;
        const unsigned long long* row = s_best + (size_t)i * a.R;
        unsigned long long run = 0ull;
        for (int r = a.R - 1; r >= 0; --r) {
            run = row[r] > run ? row[r] : run;
            a.precision[((size_t)t * a.R + r) * a.nc * cstride + pbase + m] = __longlong_as_double((long long)run);
        }
    }
}

}  // namespace yb

extern "C" int yb_coco_match(const float* boxes, const float* scores, const int64_t* classes, const int64_t* keep,
                             const int* n_keep, int B, int cap, int max_det, const double* labels, const int* n_gt,
                             const double* letterbox, int max_gt, int nc, const double* iou_thr, int T,
                             const double* area_rng, int A, yb_coco_record* records, long long* gt_count, int* status,
                             void* stream) {
    using namespace yb;
    YB_CHECK_ARG(B >= 0 && cap >= 0 && max_det >= 0 && nc >= 1, "coco_match: bad B/cap/max_det/nc");
    YB_CHECK_ARG(T >= 1 && T <= YB_MAP_MAX_T, "coco_match: 1 <= T <= %d thresholds", YB_MAP_MAX_T);
    YB_CHECK_ARG(A >= 1 && A <= YB_COCO_MAX_A && area_rng, "coco_match: 1 <= A <= %d area ranges", YB_COCO_MAX_A);
    YB_CHECK_ARG(max_gt >= 0 && max_gt <= YB_MAP_MAX_GT, "coco_match: max_gt must be in [0, %d]", YB_MAP_MAX_GT);
    if (B == 0) return 0;
    const int slots = max_det < cap ? max_det : cap;
    YB_CHECK_ARG(n_keep && n_gt && letterbox && iou_thr && gt_count && status && (slots == 0 || records),
                 "coco_match: null pointer");
    YB_CHECK_ARG(cap == 0 || (boxes && scores && classes && keep && aligned16(boxes)), "coco_match: null or unaligned candidates");
    YB_CHECK_ARG(max_gt == 0 || labels, "coco_match: null labels");
    CocoMatchArgs a{reinterpret_cast<const float4*>(boxes), scores, classes, keep, n_keep, labels, n_gt, letterbox, iou_thr,
                    records, reinterpret_cast<unsigned long long*>(gt_count), status, {}, cap, slots, max_gt, nc, T, A};
    for (int i = 0; i < 2 * A; ++i) a.rng[i] = area_rng[i];
    const int threads = T * 32 < 128 ? 128 : T * 32;
    const size_t smem = (size_t)max_gt * (sizeof(GtBox) + 2 * sizeof(int)) +
                        (size_t)threads * (sizeof(float4) + 6 * sizeof(int)) +
                        (size_t)T * ((max_gt + 31) / 32) * sizeof(unsigned int) + (size_t)nc * sizeof(int);
    YB_CHECK_ARG(smem <= (size_t)max_smem_optin(), "coco_match: %zu bytes of shared memory (nc = %d, max_gt = %d) exceed one CTA",
                 smem, nc, max_gt);
    if (smem > 48 * 1024) YB_CUDA(cudaFuncSetAttribute(coco_match_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    cudaStream_t st = (cudaStream_t)stream;
    YB_LAUNCH("coco_match_kernel", st, coco_match_kernel<<<dim3(B, A), threads, smem, st>>>(a));
    return 0;
}

extern "C" int yb_coco_precision(const yb_coco_record* records, const long long* seg, const long long* gt_count, int nc,
                                 int A, int T, const double* recall_thr, int R, const int* max_dets, int M,
                                 double* precision, double* recall, int* status, void* stream) {
    using namespace yb;
    YB_CHECK_ARG(nc >= 1 && T >= 1 && T <= YB_MAP_MAX_T && R >= 1, "coco_precision: bad nc/T/R");
    YB_CHECK_ARG(A >= 1 && A <= YB_COCO_MAX_A, "coco_precision: 1 <= A <= %d area ranges", YB_COCO_MAX_A);
    YB_CHECK_ARG(M >= 1 && M <= YB_COCO_MAX_M && max_dets, "coco_precision: 1 <= M <= %d maxDets", YB_COCO_MAX_M);
    YB_CHECK_ARG(seg && gt_count && recall_thr && precision && recall && status, "coco_precision: null pointer");
    CocoPrecArgs a{records, seg, reinterpret_cast<const unsigned long long*>(gt_count), recall_thr, precision, recall,
                   status, {}, nc, A, T, R, M};
    for (int m = 0; m < M; ++m) {
        YB_CHECK_ARG(max_dets[m] >= 1 && max_dets[m] <= 65535, "coco_precision: maxDets must be in [1, 65535], got %d",
                     max_dets[m]);
        a.max_dets[m] = max_dets[m];
    }
    const size_t smem = (size_t)M * T * R * sizeof(unsigned long long) + (size_t)R * sizeof(double);
    YB_CHECK_ARG(smem <= (size_t)max_smem_optin() - 8 * 1024, "coco_precision: T*R*M = %d*%d*%d too large for one CTA", T, R, M);
    if (smem > 48 * 1024 - 8 * 1024)
        YB_CUDA(cudaFuncSetAttribute(coco_precision_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    cudaStream_t st = (cudaStream_t)stream;
    YB_LAUNCH("coco_precision_kernel", st, coco_precision_kernel<<<dim3(nc, A), kCocoPrecThreads, smem, st>>>(a));
    return 0;
}
