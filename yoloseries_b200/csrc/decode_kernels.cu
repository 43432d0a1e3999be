// decode_kernels.cu -- the do_inference decode as ONE kernel per family: raw heads -> (b, N, C') rows.
//
// Replaces the ~12 ATen launches and three full-tensor copies per stage of trainer/eval_yolov5.py:188-209
// (and eval_yolov7.py:131-151, eval_yolox.py:135-150, eval_yolov8.py:76-102, eval_retinanet.py:59-75,
// eval_fcos.py:126-161).  This is the API-compatibility path (XEvaluator.do_inference returns the full tensor);
// the fused path (ysb_postprocess) never materialises these rows.
//
// A CTA owns 32 consecutive candidates of one image; sigmoid/exp values are produced into a shared-memory tile
// [32][C'] and written out with fully coalesced stores (32 rows of one image are contiguous in the output).
// Planes heads are read coalesced along positions (lane = candidate), rows heads along the row (lane = column).
// Templated on the head element type T: 16-bit heads are widened as they are loaded, the rows are float32.
#include "ysb_internal.cuh"

namespace ysb {

constexpr int kDecThreads = 256;
// Independent class-logit loads a thread issues before its first sigmoid.  The kernel is bound by memory-level
// parallelism: measured on B200, 64 YOLOv5s images (profiles/r2_decode_bench.txt): 4 in flight 0.330 ms, 10: 0.240 ms,
// 20: 0.217 ms for the planes layout (80 classes = 2 phases x 2 batches of 20); channels-last rows have 8 threads per row,
// i.e. 10 classes per thread at C = 80, and are fastest with exactly that batch (0.270 ms; 20 would always take the
// bounds-checked tail).
constexpr int kDecInFlight = 20;
constexpr int kDecInFlightRows = 10;

// Address of class logit 0 of a candidate and the stride between consecutive classes (hoisted out of the class loop:
// the level lookup and the two integer divisions are per candidate, not per element).
template <typename T>
struct CandAddr {
    const T *cls;
    size_t cstride;
    const T *obj;  // objectness / centerness / conf logit, nullptr when the family has none
};

template <typename T, bool NHWC>
__device__ __forceinline__ CandAddr<T> cand_addr(const Plan &P, int img, int cand)
{
    CandAddr<T> c;
    const int l = find_level(P, cand);
    const LevelDesc &lv = P.lv[l];
    const int r = cand - lv.cand_off;
    c.obj = nullptr;
    bool planes = P.layout == LAYOUT_PLANES;
    if constexpr (NHWC) planes = true;
    if (planes) {   // planes-family raw heads, NCHW or NHWC
        const int a = r / lv.hw, pos = r - a * lv.hw;
        c.cls = head_elem<T, NHWC>(lv, lv.p0, P.A, P.cls_nch, img, a, pos, P.cls_ch);
        c.cstride = static_cast<size_t>(head_step<NHWC>(lv));
        if (P.obj_col >= 0) c.obj = head_elem<T, NHWC>(lv, P.obj_src == 2 ? lv.p2 : lv.p0, P.A, P.obj_nch, img, a, pos, P.obj_ch);
    } else {
        const T *row = head_ptr<T>(lv.p0) + (static_cast<size_t>(img) * lv.img_rows + r) * P.row_w_in;
        c.cls = row + P.cls_col_in;
        c.cstride = 1;
        if (P.obj_col >= 0)
            c.obj = P.obj_src == 1 ? head_ptr<T>(P.lv[0].p1) + (static_cast<size_t>(img) * P.N + cand) * P.reg_row_w + 4 : row + P.obj_col_in;
    }
    return c;
}

// ROWS = candidates per CTA: 32 for channels-last heads (their rows are contiguous anyway; NHWC planes-family heads take
// the rows branch: cand_addr gives class step 1 and decode_box_cols reads their boxes), 128 for NCHW planes so that
// every plane access of a CTA covers 512 contiguous bytes; 16 for rows whose [32][row_w] tile exceeds the launcher's
// 200 KB (more than ~1596 classes), with 16 threads per row in the rows branch.
template <int ROWS, typename T, bool NHWC>
__global__ void __launch_bounds__(kDecThreads) k_decode_rows(const __grid_constant__ Plan P, float *__restrict__ out,
                                                              int64_t rows_total, int64_t row_offset)
{
    extern __shared__ __align__(16) float tile[];  // [ROWS][row_w]
    const int img = blockIdx.y;
    const int c0 = blockIdx.x * ROWS;
    const int nrows = min(ROWS, P.N - c0);
    const int rw = P.row_w;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (P.layout == LAYOUT_PLANES) {   // (NHWC plans: LAYOUT_ROWS_NHWC, the rows branch)
        // thread = (candidate, class phase): consecutive threads take consecutive positions of one plane
        constexpr int kPhases = kDecThreads / ROWS;  // 2 for ROWS = 128
        const int rr = threadIdx.x % ROWS, ph = threadIdx.x / ROWS;
        if (rr < nrows) {
            const CandAddr<T> ca = cand_addr<T, NHWC>(P, img, c0 + rr);
            float *tc = tile + rr * rw + P.cls_col;
            const size_t step = static_cast<size_t>(kPhases) * ca.cstride;
            // kDecInFlight independent loads per thread before the first sigmoid: the kernel is bound by memory-level
            // parallelism, not by instruction issue (4 loads in flight left DRAM at 37 % of peak)
            const float ov = (ph == 0 && ca.obj) ? ldg_head(ca.obj) : 0.0f;
            const T *src = ca.cls + static_cast<size_t>(ph) * ca.cstride;
            int k = ph;
            // whole batches need no per-load bounds test (80 classes: four of them)
            for (; k + (kDecInFlight - 1) * kPhases < P.C; k += kDecInFlight * kPhases, src += kDecInFlight * step) {
                float v[kDecInFlight];
#pragma unroll
                for (int u = 0; u < kDecInFlight; ++u) v[u] = ldg_head(src + u * step);
                bool redo = false;
#pragma unroll
                for (int u = 0; u < kDecInFlight; ++u) tc[k + u * kPhases] = sigmoid_fast(v[u], redo);
                if (__builtin_expect(redo, 0)) {   // a logit below -87.3: denormal sigmoid, library reciprocal
#pragma unroll
                    for (int u = 0; u < kDecInFlight; ++u) tc[k + u * kPhases] = sigmoid_ref(v[u]);
                }
            }
            if (k < P.C) {
                float v[kDecInFlight];
#pragma unroll
                for (int u = 0; u < kDecInFlight; ++u) v[u] = (k + u * kPhases < P.C) ? ldg_head(src + u * step) : 0.0f;
#pragma unroll
                for (int u = 0; u < kDecInFlight; ++u)
                    if (k + u * kPhases < P.C) tc[k + u * kPhases] = sigmoid_ref(v[u]);
            }
            if (ph == 0 && ca.obj) tile[rr * rw + P.obj_col] = sigmoid_ref(ov);
        }
        if (P.family == YSB_YOLOV8) {
            // DFL boxes: four threads per candidate (one side each), 64 candidates per round
            for (int base = 0; base < nrows; base += kDecThreads / 4) {
                const int r4 = base + (threadIdx.x >> 2), side = threadIdx.x & 3;
                float sv = 0.0f;
                if (r4 < nrows) sv = v8_side_value<T, NHWC>(P, img, c0 + r4, side);
                const unsigned qb = lane & ~3u;
                const float s0 = __shfl_sync(0xffffffffu, sv, qb), s1 = __shfl_sync(0xffffffffu, sv, qb + 1);
                const float s2 = __shfl_sync(0xffffffffu, sv, qb + 2), s3 = __shfl_sync(0xffffffffu, sv, qb + 3);
                if (side == 0 && r4 < nrows) {
                    const float4 b = tta_undo(P, v8_box_from_sides(P, c0 + r4, s0, s1, s2, s3));
                    float *t = tile + r4 * rw + P.box_col;
                    t[0] = b.x; t[1] = b.y; t[2] = b.z; t[3] = b.w;
                }
            }
        } else if (threadIdx.x >= kDecThreads - ROWS && threadIdx.x - (kDecThreads - ROWS) < nrows) {
            const int rb = threadIdx.x - (kDecThreads - ROWS);
            const float4 b = tta_undo(P, decode_box_cols<T, NHWC>(P, img, c0 + rb));
            float *t = tile + rb * rw + P.box_col;
            t[0] = b.x; t[1] = b.y; t[2] = b.z; t[3] = b.w;
        }
    } else {
        // eight threads per candidate row (32 rows x 8): a warp reads 4 rows x 32 contiguous bytes per step, every
        // fetched sector fully used; kDecInFlightRows loads in flight per thread.  Lane-per-candidate box / objectness decode.
        constexpr int TPR = ROWS >= 32 ? 8 : kDecThreads / ROWS;   // threads per row
        const int r = threadIdx.x / TPR, q = threadIdx.x % TPR;
        if (r < nrows) {
            const CandAddr<T> ca = cand_addr<T, NHWC>(P, img, c0 + r);
            float *tc = tile + r * rw + P.cls_col;
            int k = q;
            for (; k + TPR * (kDecInFlightRows - 1) < P.C; k += TPR * kDecInFlightRows) {
                float v[kDecInFlightRows];
#pragma unroll
                for (int u = 0; u < kDecInFlightRows; ++u) v[u] = ldg_head(ca.cls + k + TPR * u);
                bool redo = false;
#pragma unroll
                for (int u = 0; u < kDecInFlightRows; ++u) tc[k + TPR * u] = sigmoid_fast(v[u], redo);
                if (__builtin_expect(redo, 0)) {
#pragma unroll
                    for (int u = 0; u < kDecInFlightRows; ++u) tc[k + TPR * u] = sigmoid_ref(v[u]);
                }
            }
            if (k < P.C) {
                float v[kDecInFlightRows];
#pragma unroll
                for (int u = 0; u < kDecInFlightRows; ++u) v[u] = (k + TPR * u < P.C) ? ldg_head(ca.cls + k + TPR * u) : 0.0f;
#pragma unroll
                for (int u = 0; u < kDecInFlightRows; ++u)
                    if (k + TPR * u < P.C) tc[k + TPR * u] = sigmoid_ref(v[u]);
            }
        }
        if (warp == 0 && lane < nrows) {
            const int cand = c0 + lane;
            const float4 b = tta_undo(P, decode_box_cols<T, NHWC>(P, img, cand));
            float *t = tile + lane * rw + P.box_col;
            t[0] = b.x; t[1] = b.y; t[2] = b.z; t[3] = b.w;
            if (P.obj_col >= 0) {
                const CandAddr<T> ca = cand_addr<T, NHWC>(P, img, cand);
                t[P.obj_col - P.box_col] = sigmoid_ref(ldg_head(ca.obj));
            }
        }
    }
    __syncthreads();
    float *dst = out + (static_cast<size_t>(img) * rows_total + row_offset + c0) * rw;
    const int nfl = nrows * rw;
    if (((reinterpret_cast<uintptr_t>(dst) | reinterpret_cast<uintptr_t>(tile)) & 15u) == 0) {
        const int nv = nfl >> 2;
        for (int e = threadIdx.x; e < nv; e += kDecThreads)
            reinterpret_cast<float4 *>(dst)[e] = reinterpret_cast<const float4 *>(tile)[e];
        for (int e = (nv << 2) + threadIdx.x; e < nfl; e += kDecThreads) dst[e] = tile[e];
    } else {
        for (int e = threadIdx.x; e < nfl; e += kDecThreads) dst[e] = tile[e];
    }
}

template <int ROWS, typename T, bool NHWC = false>
static cudaError_t launch_decode_t(const Plan &P, float *d_out, int64_t rows_total, int64_t row_offset, cudaStream_t stream)
{
    const size_t smem = static_cast<size_t>(ROWS) * P.row_w * sizeof(float);
    if (smem > 200 * 1024) return cudaErrorInvalidValue;
    if (smem > 48 * 1024) {
        cudaError_t e = cudaFuncSetAttribute(k_decode_rows<ROWS, T, NHWC>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
        if (e != cudaSuccess) return e;
    }
    const dim3 grid((P.N + ROWS - 1) / ROWS, P.batch);
    k_decode_rows<ROWS, T, NHWC><<<grid, kDecThreads, smem, stream>>>(P, d_out, rows_total, row_offset);
    return cudaGetLastError();
}

template <typename T>
static cudaError_t launch_decode_dt(const Plan &P, float *d_out, int64_t rows_total, int64_t row_offset, cudaStream_t stream)
{
    if (P.layout == LAYOUT_ROWS_NHWC) return launch_decode_t<32, T, true>(P, d_out, rows_total, row_offset, stream);   // rows branch, 32 rows / CTA
    if (P.layout == LAYOUT_PLANES && static_cast<size_t>(128) * P.row_w * sizeof(float) <= 100 * 1024)
        return launch_decode_t<128, T>(P, d_out, rows_total, row_offset, stream);
    if (static_cast<size_t>(32) * P.row_w * sizeof(float) <= 200 * 1024) return launch_decode_t<32, T>(P, d_out, rows_total, row_offset, stream);
    return launch_decode_t<16, T>(P, d_out, rows_total, row_offset, stream);   // rows of more than 1600 values
}

// rows_total / row_offset: the pass fills rows [row_offset, row_offset + N) of a (batch, rows_total, C') tensor
cudaError_t launch_decode(const Plan &P, float *d_out, int64_t rows_total, int64_t row_offset, cudaStream_t stream,
                          int dtype)
{
    if (P.batch == 0 || P.N == 0) return cudaSuccess;
    switch (dtype) {
    case YSB_F16: return launch_decode_dt<__half>(P, d_out, rows_total, row_offset, stream);
    case YSB_BF16: return launch_decode_dt<__nv_bfloat16>(P, d_out, rows_total, row_offset, stream);
    default: return launch_decode_dt<float>(P, d_out, rows_total, row_offset, stream);
    }
}

// Self-test: the spelled-out reciprocal of sigmoid_ref / sigmoid_fast against __frcp_rn for EVERY float in [1, +inf]
// (bit patterns 0x3f800000 .. 0x7f800000, 1.07e9 values).  mismatches[0] += values where rcp_rn_ge1 differs,
// mismatches[1] += values below 2^126 where the branch-free fast path differs or flags a redo, or at / above 2^126 where
// it fails to flag one.
__global__ void __launch_bounds__(256) k_selftest_reciprocal(unsigned long long *__restrict__ mismatches)
{
    const uint32_t lo = 0x3f800000u, hi = 0x7f800000u;
    unsigned long long bad0 = 0, bad1 = 0;
    for (uint64_t b = lo + static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x; b <= hi;
         b += static_cast<uint64_t>(gridDim.x) * blockDim.x) {
        const float d = __uint_as_float(static_cast<uint32_t>(b));
        const uint32_t want = __float_as_uint(__frcp_rn(d));
        if (__float_as_uint(rcp_rn_ge1(d)) != want) ++bad0;
        float r;
        asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(d));
        const float e = __fmaf_rn(d, r, -1.0f);
        const uint32_t fast = __float_as_uint(__fmaf_rn(r, -e, r));
        const bool redo = d >= 8.507059173e37f;
        if (redo != (b >= 0x7e800000u) || (!redo && fast != want)) ++bad1;
    }
    if (bad0) atomicAdd(mismatches, bad0);
    if (bad1) atomicAdd(mismatches + 1, bad1);
}

cudaError_t launch_selftest_reciprocal(unsigned long long *d_mismatches, cudaStream_t stream)
{
    cudaError_t e = cudaMemsetAsync(d_mismatches, 0, 2 * sizeof(unsigned long long), stream);
    if (e != cudaSuccess) return e;
    k_selftest_reciprocal<<<148 * 8, 256, 0, stream>>>(d_mismatches);
    return cudaGetLastError();
}

}  // namespace ysb
