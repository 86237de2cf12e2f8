// yb_decode.cu — K1 / K1b: decode_predictions forward and its vector-Jacobian product.
// Reference: train.py:712-779.  Bound: HBM (read T + write T forward; read 2T + write T backward).
//
// Layout: the head tensor is one contiguous fp32, bf16 or fp16 array of B*H*W*A rows of (5+nc) elements.
// The kernels walk it as flat 16-byte vectors (4 floats or 8 halves) — fully coalesced for any nc — and
// recover (row, channel) with an exact multiply-shift division; only channels 0..3 of a row do
// arithmetic, everything else is a straight copy.
#include "yb_common.cuh"

namespace yb {

struct DecodeArgs {
    const void* pred;       // element type T of the kernel (float, bf16, fp16)
    const float* anchors;   // (A,2) device
    const void* grad_out;   // bwd only
    void* out;              // fwd: decoded; bwd: grad_in
    uint32_t n_vec;         // number of whole 16-byte vectors
    uint32_t n_elem;        // total elements
    uint32_t row;           // 5+nc
    int A, W, H;
    FastDiv d_row, d_A, d_W, d_H;
    DecodeConsts k;
};

template <bool BWD>
__device__ __forceinline__ float decode_elem(const DecodeArgs& a, uint32_t r, uint32_t c, float x, float g) {
    // r = flat row index ((b*H + gy)*W + gx)*A + an ; c = channel in row
    if (c >= 4) return BWD ? g : x;
    uint32_t cell, an, gy_b, gx, gy, bi;
    a.d_A.divmod(r, cell, an);
    a.d_W.divmod(cell, gy_b, gx);
    a.d_H.divmod(gy_b, bi, gy);
    if (!BWD) {
        if (c == 0) return decode_xy(x, (float)gx, a.k.inv_w);
        if (c == 1) return decode_xy(x, (float)gy, a.k.inv_h);
        float anc = __ldg(a.anchors + an * 2 + (c - 2));
        return decode_wh(x, anc, a.k.inv_img);
    } else {
        // autograd order of train.py:758-759,773-774 (see DESIGN.md "decode backward")
        float s = sigmoidf_ref(x);
        float ds = (1.0f - s) * s;  // sigmoid_backward: grad * ((1 - y) * y)
        if (c < 2) {
            float inv = (c == 0) ? a.k.inv_w : a.k.inv_h;
            return ((g * inv) * 2.0f) * ds;
        }
        float anc = __ldg(a.anchors + an * 2 + (c - 2));
        float u = 2.0f * s;
        float gp = g * (anc * a.k.inv_img);  // mul backward
        float gu = gp * (2.0f * u);          // pow(u,2) backward
        return (gu * 2.0f) * ds;             // (2*s) backward, then sigmoid backward
    }
}

// element e of the flat head tensor, widened, decoded and rounded back (tails of the vector walks)
template <typename T, bool BWD>
__device__ __forceinline__ void decode_one(const DecodeArgs& a, uint32_t e) {
    uint32_t r, c;
    a.d_row.divmod(e, r, c);
    const T* x = reinterpret_cast<const T*>(a.pred);
    const T* g = reinterpret_cast<const T*>(a.grad_out);
    reinterpret_cast<T*>(a.out)[e] = from_f32<T>(decode_elem<BWD>(a, r, c, to_f32(x[e]), BWD ? to_f32(g[e]) : 0.f));
}

template <typename T, bool BWD>
__global__ void __launch_bounds__(256) decode_kernel(const DecodeArgs a) {
    constexpr uint32_t V = kVec<T>;
    const uint32_t stride = gridDim.x * blockDim.x;
    const float4* __restrict__ in4 = reinterpret_cast<const float4*>(a.pred);
    const float4* __restrict__ g4 = reinterpret_cast<const float4*>(a.grad_out);
    float4* __restrict__ out4 = reinterpret_cast<float4*>(a.out);
    for (uint32_t v = blockIdx.x * blockDim.x + threadIdx.x; v < a.n_vec; v += stride) {
        float4 x = __ldcs(in4 + v);
        float4 g = BWD ? __ldcs(g4 + v) : make_float4(0.f, 0.f, 0.f, 0.f);
        uint32_t r, c;
        a.d_row.divmod(v * V, r, c);
        if (c >= 4u && c + (V - 1u) < a.row) {   // V logits of one row (81 of 85 floats at nc=80): a straight copy
            __stcs(out4 + v, BWD ? g : x);
            continue;
        }
        float xs[V], gs[V], o[V];
        unpack16<T>(x, xs);
        unpack16<T>(g, gs);
#pragma unroll
        for (int k = 0; k < (int)V; ++k) {
            o[k] = decode_elem<BWD>(a, r, c, xs[k], gs[k]);
            if (++c == a.row) { c = 0; ++r; }
        }
        __stcs(out4 + v, pack16<T>(o));
    }
    // scalar tail (n_elem not a multiple of V)
    if (blockIdx.x == 0 && threadIdx.x < a.n_elem % V) decode_one<T, BWD>(a, a.n_vec * V + threadIdx.x);
}

// Short rows (5..8 elements: nc <= 3, e.g. the reference's single-class 'cone' model): two thirds of the elements
// need a sigmoid, so the flat walk's per-element (row, channel) bookkeeping costs as much as the arithmetic.  Here a
// thread owns R = V/gcd(ROW,V) whole rows = ROW*R/V 16-byte vectors (V = 4 floats or 8 halves; still fully coalesced:
// consecutive threads own consecutive segments), decomposes the row index once per row and runs straight-line code.
__host__ __device__ constexpr int gcd_c(int a, int b) { return b == 0 ? a : gcd_c(b, a % b); }
template <int ROW, typename T, bool BWD>
__global__ void __launch_bounds__(256) decode_rows_kernel(const DecodeArgs a) {
    constexpr int V = (int)kVec<T>;
    constexpr int R = V / gcd_c(ROW, V);
    constexpr int NV = ROW * R / V;
    const uint32_t n_groups = a.n_elem / (uint32_t)(ROW * R);   // whole groups; the remainder rows go to the tail below
    const uint32_t stride = gridDim.x * blockDim.x;
    const float4* __restrict__ in4 = reinterpret_cast<const float4*>(a.pred);
    const float4* __restrict__ g4 = reinterpret_cast<const float4*>(a.grad_out);
    float4* __restrict__ out4 = reinterpret_cast<float4*>(a.out);
    for (uint32_t gidx = blockIdx.x * blockDim.x + threadIdx.x; gidx < n_groups; gidx += stride) {
        float x[NV * V], g[NV * V], o[NV * V];
#pragma unroll
        for (int v = 0; v < NV; ++v) {
            unpack16<T>(__ldcs(in4 + (size_t)gidx * NV + v), x + V * v);
            if (BWD) unpack16<T>(__ldcs(g4 + (size_t)gidx * NV + v), g + V * v);
        }
#pragma unroll
        for (int k = 0; k < R; ++k) {
            const uint32_t r = gidx * R + k;
            uint32_t cell, an, gy_b, gx, gy, bi;
            a.d_A.divmod(r, cell, an);
            a.d_W.divmod(cell, gy_b, gx);
            a.d_H.divmod(gy_b, bi, gy);
            const float aw = __ldg(a.anchors + an * 2), ah = __ldg(a.anchors + an * 2 + 1);
            const float* xr = x + k * ROW;
            float* orow = o + k * ROW;
            if (!BWD) {
                orow[0] = decode_xy(xr[0], (float)gx, a.k.inv_w);
                orow[1] = decode_xy(xr[1], (float)gy, a.k.inv_h);
                orow[2] = decode_wh(xr[2], aw, a.k.inv_img);
                orow[3] = decode_wh(xr[3], ah, a.k.inv_img);
#pragma unroll
                for (int c = 4; c < ROW; ++c) orow[c] = xr[c];
            } else {
                const float* gr = g + k * ROW;
#pragma unroll
                for (int c = 0; c < 4; ++c) {   // autograd order of train.py:758-759,773-774, as in decode_elem
                    const float s = sigmoidf_ref(xr[c]);
                    const float ds = (1.0f - s) * s;
                    if (c < 2) {
                        orow[c] = ((gr[c] * (c == 0 ? a.k.inv_w : a.k.inv_h)) * 2.0f) * ds;
                    } else {
                        const float u = 2.0f * s;
                        const float gp = gr[c] * ((c == 2 ? aw : ah) * a.k.inv_img);
                        orow[c] = ((gp * (2.0f * u)) * 2.0f) * ds;
                    }
                }
#pragma unroll
                for (int c = 4; c < ROW; ++c) orow[c] = gr[c];
            }
        }
#pragma unroll
        for (int v = 0; v < NV; ++v) __stcs(out4 + (size_t)gidx * NV + v, pack16<T>(o + V * v));
    }
    // the last (< R) rows
    const uint32_t e0 = n_groups * (uint32_t)(ROW * R);
    if (blockIdx.x == 0 && e0 + threadIdx.x < a.n_elem) decode_one<T, BWD>(a, e0 + threadIdx.x);
}

// The four box channels of row r from their sigmoids s[0..3] (sigmoid_ref_batch): forward values, or the
// vector-Jacobian product with the upstream gradients gr[0..3] — the same expressions as decode_elem.
template <bool BWD>
__device__ __forceinline__ void decode_row4(const DecodeArgs& a, uint32_t r, const float* s, const float* gr, float* orow) {
    uint32_t cell, an, gy_b, gx, gy, bi;
    a.d_A.divmod(r, cell, an);
    a.d_W.divmod(cell, gy_b, gx);
    a.d_H.divmod(gy_b, bi, gy);
    const float aw = __ldg(a.anchors + an * 2), ah = __ldg(a.anchors + an * 2 + 1);
    if (!BWD) {
        orow[0] = decode_xy_s(s[0], (float)gx, a.k.inv_w);
        orow[1] = decode_xy_s(s[1], (float)gy, a.k.inv_h);
        orow[2] = decode_wh_s(s[2], aw, a.k.inv_img);
        orow[3] = decode_wh_s(s[3], ah, a.k.inv_img);
    } else {
#pragma unroll
        for (int c = 0; c < 4; ++c) {   // autograd order of train.py:758-759,773-774, as in decode_elem
            const float ds = (1.0f - s[c]) * s[c];
            if (c < 2) {
                orow[c] = ((gr[c] * (c == 0 ? a.k.inv_w : a.k.inv_h)) * 2.0f) * ds;
            } else {
                const float u = 2.0f * s[c];
                const float gp = gr[c] * ((c == 2 ? aw : ah) * a.k.inv_img);
                orow[c] = ((gp * (2.0f * u)) * 2.0f) * ds;
            }
        }
    }
}

// Long rows (nc >= 4, e.g. 85 floats): in the flat walk a quarter of the lanes of every warp holds one of a row's
// four box channels, so every warp ran the full sigmoid path (300 instructions per float4, ncu: 247 M warp
// instructions for the 418 MB P3 head, 0.48 of the copy peak).  Here a CTA owns 64 consecutive rows (a 16-byte
// aligned span for any row length and element size): phase 1 is a pure 16-byte copy of the span, phase 2 — after a
// barrier — lets one thread per row overwrite the four box channels with the decoded values (the sectors are still
// in L2).  That thread decomposes its row index once and evaluates its four sigmoids in ONE basic block
// (sigmoid_ref_batch: the division's branch to its slow path made them four serial chains, and only 64 of the CTA's
// 256 threads work in this phase): nc=80, B=64, 640^2: forward 248 -> 225 us, backward 330 -> 235 us.  (In the
// short-row kernel above the same batching changed nothing forward and cost registers backward: 15.0 -> 16.3 us on
// the P3 head; not adopted there.)
template <typename T, bool BWD>
__global__ void __launch_bounds__(256) decode_long_kernel(const DecodeArgs a) {
    constexpr uint32_t RPC = 64;   // rows per chunk (64*row elements is a multiple of 16 bytes)
    const T* __restrict__ pred = reinterpret_cast<const T*>(a.pred);
    const T* __restrict__ grad_out = reinterpret_cast<const T*>(a.grad_out);
    T* __restrict__ out = reinterpret_cast<T*>(a.out);
    const uint32_t n_rows = a.n_elem / a.row;
    const uint32_t n_chunks = (n_rows + RPC - 1) / RPC;
    for (uint32_t ch = blockIdx.x; ch < n_chunks; ch += gridDim.x) {
        const uint32_t r0 = ch * RPC, nr = min(RPC, n_rows - r0);
        const size_t e0 = (size_t)r0 * a.row;
        const uint32_t nfl = nr * a.row, nv = nfl / kVec<T>;
        const float4* __restrict__ src4 = reinterpret_cast<const float4*>((BWD ? grad_out : pred) + e0);
        float4* __restrict__ dst4 = reinterpret_cast<float4*>(out + e0);
        for (uint32_t v0 = threadIdx.x; v0 < nv; v0 += 6 * 256) {   // six independent 16-byte loads in flight per thread
            float4 t[6];
#pragma unroll
            for (int k = 0; k < 6; ++k) if (v0 + k * 256 < nv) t[k] = __ldcs(src4 + v0 + k * 256);
#pragma unroll
            for (int k = 0; k < 6; ++k) if (v0 + k * 256 < nv) __stcg(dst4 + v0 + k * 256, t[k]);
        }
        for (uint32_t e = nv * kVec<T> + threadIdx.x; e < nfl; e += 256) out[e0 + e] = (BWD ? grad_out : pred)[e0 + e];
        __syncthreads();
        if (threadIdx.x < nr) {
            const uint32_t r = r0 + threadIdx.x;
            const size_t eb = (size_t)r * a.row;
            float xr[4], gr[4] = {0.f, 0.f, 0.f, 0.f}, sg[4], o[4];
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                xr[c] = to_f32(pred[eb + c]);
                if (BWD) gr[c] = to_f32(grad_out[eb + c]);
            }
            sigmoid_ref_batch<4>(xr, sg);
            decode_row4<BWD>(a, r, sg, gr, o);
#pragma unroll
            for (int c = 0; c < 4; ++c) out[eb + c] = from_f32<T>(o[c]);
        }
        __syncthreads();
    }
}

template <int ROW, typename T>
static void decode_rows_launch(bool bwd, const DecodeArgs& a, int blocks, cudaStream_t st) {
    if (bwd) decode_rows_kernel<ROW, T, true><<<blocks, 256, 0, st>>>(a);
    else     decode_rows_kernel<ROW, T, false><<<blocks, 256, 0, st>>>(a);
}

template <typename T>
static int decode_launch_t(bool bwd, const DecodeArgs& a, unsigned long long n, cudaStream_t st) {
    const int threads = 256;
    unsigned long long want = ((unsigned long long)a.n_vec + threads - 1) / threads;
    // 8 resident CTAs/SM x 148 SMs, grid-stride beyond that (multiple of the SM count)
    unsigned long long cap = (unsigned long long)sm_count() * 8 * 4;
    int blocks = (int)(want < 1 ? 1 : (want < cap ? want : cap));
    const char* name = bwd ? "decode_bwd_kernel" : "decode_fwd_kernel";
    if (a.row <= 8) {   // short rows: whole rows per thread
        const unsigned long long V = kVec<T>;
        unsigned long long R = V;
        while (R > 1 && (a.row * R / 2) % V == 0) R /= 2;   // V / gcd(row, V), V a power of two
        unsigned long long groups = n / (a.row * R);
        unsigned long long w2 = (groups + threads - 1) / threads;
        blocks = (int)(w2 < 1 ? 1 : (w2 < cap ? w2 : cap));
        switch (a.row) {
            case 5: YB_LAUNCH(name, st, decode_rows_launch<5, T>(bwd, a, blocks, st)); break;
            case 6: YB_LAUNCH(name, st, decode_rows_launch<6, T>(bwd, a, blocks, st)); break;
            case 7: YB_LAUNCH(name, st, decode_rows_launch<7, T>(bwd, a, blocks, st)); break;
            default: YB_LAUNCH(name, st, decode_rows_launch<8, T>(bwd, a, blocks, st)); break;
        }
        return 0;
    }
    if (a.row >= 16) {   // long rows: copy + per-row fix-up
        unsigned long long chunks = (n / a.row + 63) / 64;
        blocks = (int)(chunks < 1 ? 1 : (chunks < cap ? chunks : cap));
        if (bwd) YB_LAUNCH(name, st, decode_long_kernel<T, true><<<blocks, threads, 0, st>>>(a));
        else     YB_LAUNCH(name, st, decode_long_kernel<T, false><<<blocks, threads, 0, st>>>(a));
        return 0;
    }
    if (bwd) YB_LAUNCH(name, st, decode_kernel<T, true><<<blocks, threads, 0, st>>>(a));
    else     YB_LAUNCH(name, st, decode_kernel<T, false><<<blocks, threads, 0, st>>>(a));
    return 0;
}

static int decode_launch(bool bwd, const void* pred, const float* anchors, const void* grad_out,
                         void* out, int B, int H, int W, int A, int nc, float img_size, int dtype,
                         void* stream) {
    YB_CHECK_ARG(pred && anchors && out && (!bwd || grad_out), "decode: null pointer");
    YB_CHECK_ARG(B >= 0 && H > 0 && W > 0 && A > 0 && A <= YB_MAX_ANCHORS && nc >= 0,
                 "decode: bad shape B=%d H=%d W=%d A=%d nc=%d", B, H, W, A, nc);
    YB_CHECK_ARG(aligned16(pred) && aligned16(out) && (!bwd || aligned16(grad_out)),
                 "decode: tensors must be 16-byte aligned");
    unsigned long long n = (unsigned long long)B * H * W * A * (5 + nc);
    YB_CHECK_ARG(n < (1ull << 32), "decode: tensor too large (%llu elements)", n);
    YB_CHECK_ARG(dtype == YB_DTYPE_F32 || dtype == YB_DTYPE_BF16 || dtype == YB_DTYPE_F16, "decode: unknown dtype %d", dtype);
    if (n == 0) return 0;
    DecodeArgs a;
    a.pred = pred; a.anchors = anchors; a.grad_out = grad_out; a.out = out;
    a.n_elem = (uint32_t)n; a.n_vec = (uint32_t)(n * dtype_size(dtype) / 16); a.row = 5 + nc;
    a.A = A; a.W = W; a.H = H;
    a.d_row = FastDiv(5 + nc); a.d_A = FastDiv(A); a.d_W = FastDiv(W); a.d_H = FastDiv(H);
    a.k.inv_w = 1.0f / (float)W; a.k.inv_h = 1.0f / (float)H; a.k.inv_img = 1.0f / img_size;
    cudaStream_t st = (cudaStream_t)stream;
    YB_DISPATCH_DTYPE(dtype, T, return decode_launch_t<T>(bwd, a, n, st));
    return 0;
}

// ---- self-test of rcp_normal / sigmoid_ref_batch (yb_selftest_sigmoid) -----------------------------------------
__global__ void __launch_bounds__(256) selftest_rcp_kernel(unsigned long long* bad) {
    const unsigned long long n = 0xfcull << 23;   // biased exponents 1..252, either sign
    unsigned long long mism = 0;
    for (unsigned long long i = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x; i < 2 * n;
         i += (unsigned long long)gridDim.x * blockDim.x) {
        const uint32_t bits = ((uint32_t)(i % n) + (1u << 23)) | (i >= n ? 0x80000000u : 0u);
        const float y = __uint_as_float(bits);
        if (__float_as_uint(1.0f / y) != __float_as_uint(rcp_normal(y))) ++mism;
    }
    if (mism) atomicAdd(bad, mism);
}
__global__ void __launch_bounds__(256) selftest_sigmoid_kernel(unsigned long long* bad) {
    unsigned long long mism = 0;
    for (unsigned long long i = (blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x) * 4ull; i < (1ull << 32);
         i += (unsigned long long)gridDim.x * blockDim.x * 4ull) {
        float x[4], s[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) x[k] = __uint_as_float((uint32_t)i + (uint32_t)k);
        sigmoid_ref_batch<4>(x, s);   // includes the fallback for values outside the fast range
#pragma unroll
        for (int k = 0; k < 4; ++k)
            if (x[k] == x[k] && __float_as_uint(sigmoidf_ref(x[k])) != __float_as_uint(s[k])) ++mism;
    }
    if (mism) atomicAdd(bad, mism);
}

}  // namespace yb

extern "C" int yb_selftest_sigmoid(unsigned long long* mismatches_host, void* stream) {
    using namespace yb;
    YB_CHECK_ARG(mismatches_host, "selftest: null output");
    cudaStream_t st = (cudaStream_t)stream;
    unsigned long long* d = nullptr;
    YB_CUDA(cudaMalloc(&d, 2 * sizeof(unsigned long long)));   // test entry point: the only allocation in the library
    cudaError_t e = cudaMemsetAsync(d, 0, 2 * sizeof(unsigned long long), st);
    if (e == cudaSuccess) {
        selftest_rcp_kernel<<<sm_count() * 8, 256, 0, st>>>(d);
        selftest_sigmoid_kernel<<<sm_count() * 8, 256, 0, st>>>(d + 1);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaMemcpyAsync(mismatches_host, d, 2 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    cudaFree(d);
    if (e != cudaSuccess) {
        set_error("yb_selftest_sigmoid failed: %s", cudaGetErrorString(e));
        return (int)e;
    }
    count_launch(2);
    return 0;
}

extern "C" int yb_decode_fwd(const float* pred, const float* anchors, float* out, int B, int H,
                             int W, int A, int nc, float img_size, void* stream) {
    return yb::decode_launch(false, pred, anchors, nullptr, out, B, H, W, A, nc, img_size, YB_DTYPE_F32, stream);
}

extern "C" int yb_decode_bwd(const float* pred, const float* anchors, const float* grad_out,
                             float* grad_in, int B, int H, int W, int A, int nc, float img_size,
                             void* stream) {
    return yb::decode_launch(true, pred, anchors, grad_out, grad_in, B, H, W, A, nc, img_size, YB_DTYPE_F32, stream);
}

extern "C" int yb_decode_fwd_t(const void* pred, const float* anchors, void* out, int B, int H, int W, int A, int nc,
                               float img_size, int dtype, void* stream) {
    return yb::decode_launch(false, pred, anchors, nullptr, out, B, H, W, A, nc, img_size, dtype, stream);
}

extern "C" int yb_decode_bwd_t(const void* pred, const float* anchors, const void* grad_out, void* grad_in, int B, int H,
                               int W, int A, int nc, float img_size, int dtype, void* stream) {
    return yb::decode_launch(true, pred, anchors, grad_out, grad_in, B, H, W, A, nc, img_size, dtype, stream);
}
