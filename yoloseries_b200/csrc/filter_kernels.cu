// filter_kernels.cu -- K1: fused (sigmoid) + filter + class pick + stream compaction.
//
// Replaces the head of every evaluator's numba_nms method (trainer/eval_yolov5.py:265-286 and the same block
// in eval_yolov7/yolox/yolov8/retinanet/retinanet_experiment/fcos; per-family operators in SURVEY.md 8a-2)
// together with the sigmoid part of do_inference for the channels that feed the score.
//
// HBM-bound streaming pass: every class/objectness logit is read exactly once (box channels are NOT read here;
// the few candidates that reach NMS get their boxes decoded in the NMS kernel).  Per candidate the kernel keeps
// the two largest class logits and the first arg-max, evaluates sigmoid only for the winner (sigmoid is
// monotone, float32 rounding is monotone) and falls back to evaluating every near-tied class exactly when the
// runner-up is within a guard band -- so score and class id are bit-identical to "sigmoid all, multiply all,
// max/argmax" as the reference does, at ~5 ALU ops per logit instead of ~25.
//
// Output: one 64-bit sort key per survivor, written with warp-aggregated atomics (order inside an image is
// irrelevant: the key carries the candidate index, see pack_key).
//
// Every kernel is templated on the head element type T (float, __half, __nv_bfloat16): values are widened to float32 as
// they are loaded, so survivors, scores and classes are those of the float32 path on the widened heads.  The float
// instantiations are the kernels of the float32-only engine, unchanged.
//
// Kernels in this file (dispatch: launch_filter at the bottom):
//   k_filter_planes_v4     NCHW heads whose levels are all 128-bit loadable (YOLOv5 / YOLOX / YOLOv8)   -- product path
//   k_filter_planes        NCHW heads with levels that are not (FCOS' 5x5 map); generic                   -- product path
//   k_filter_rows          channels-last heads and the decoded (b, N, C') tensor (YOLOv7, RetinaNet; NHWC  -- product path
//                          YOLOv5 / YOLOX / YOLOv8 / FCOS heads through its NHWC instantiation)
//   k_filter_multilabel    hyp['mutil_label']: one key per (candidate, class)                              -- product path
// The cp.async ring, 1-D bulk-copy TMA ring and 2-D tensor-map TMA ring variants that were measured against these (same
// survivor sets, slower on this access pattern; profiles/README.md) live in filter_variants.cuh and are compiled only with
// -DYSB_PROFILING_VARIANTS: the product library has exactly one kernel per layout and no environment switches.
#ifdef YSB_PROFILING_VARIANTS
#include <cuda.h>
#endif

#include <cstdlib>
#include <cstring>

#include "ysb_internal.cuh"

namespace ysb {

__device__ __forceinline__ float4 ldg_stream4(const float *p)
{
    float4 v;
    asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
                 : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
                 : "l"(p));
    return v;
}
__device__ __forceinline__ float4 ldg_stream4_256(const float *p)
{
    float4 v;
    asm volatile("ld.global.nc.L1::no_allocate.L2::256B.v4.f32 {%0,%1,%2,%3}, [%4];"
                 : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
                 : "l"(p));
    return v;
}
__device__ __forceinline__ float ldg_stream1(const float *p)
{
    float v;
    asm volatile("ld.global.nc.L1::no_allocate.f32 %0, [%1];" : "=f"(v) : "l"(p));
    return v;
}

// 16-bit heads: four consecutive values are one 64-bit load (a warp reads 256 contiguous bytes per class plane), widened
// to the float4 the float32 kernels work on.  Element 0 is the low half of the first word (little endian).
__device__ __forceinline__ float4 widen4(uint2 r, const __half *)
{
    return make_float4(__half2float(__ushort_as_half(static_cast<unsigned short>(r.x & 0xffffu))),
                       __half2float(__ushort_as_half(static_cast<unsigned short>(r.x >> 16))),
                       __half2float(__ushort_as_half(static_cast<unsigned short>(r.y & 0xffffu))),
                       __half2float(__ushort_as_half(static_cast<unsigned short>(r.y >> 16))));
}
__device__ __forceinline__ float4 widen4(uint2 r, const __nv_bfloat16 *)
{
    return make_float4(__uint_as_float(r.x << 16), __uint_as_float(r.x & 0xffff0000u), __uint_as_float(r.y << 16),
                       __uint_as_float(r.y & 0xffff0000u));
}
template <typename T>
__device__ __forceinline__ float4 ldg_stream4(const T *p)
{
    uint2 r;
    asm volatile("ld.global.nc.L1::no_allocate.v2.u32 {%0,%1}, [%2];" : "=r"(r.x), "=r"(r.y) : "l"(p));
    return widen4(r, p);
}
template <typename T>
__device__ __forceinline__ float4 ldg_stream4_256(const T *p)
{
    uint2 r;
    asm volatile("ld.global.nc.L1::no_allocate.L2::256B.v2.u32 {%0,%1}, [%2];" : "=r"(r.x), "=r"(r.y) : "l"(p));
    return widen4(r, p);
}
// one raw 16-bit element (staged unconverted into the rows kernel's tile)
template <typename T>
__device__ __forceinline__ T ldg_stream1_raw(const T *p)
{
    unsigned short v;
    asm volatile("ld.global.nc.L1::no_allocate.u16 %0, [%1];" : "=h"(v) : "l"(p));
    return *reinterpret_cast<const T *>(&v);
}
__device__ __forceinline__ float ldg_stream1_raw(const float *p) { return ldg_stream1(p); }
template <typename T>
__device__ __forceinline__ float ldg_stream1(const T *p) { return widen(ldg_stream1_raw(p)); }

__device__ __forceinline__ void top2_update(float c, int k, float &m1, float &m2, int &k0)
{
    m2 = fmaxf(m2, fminf(m1, c));
    k0 = (c > m1) ? k : k0;
    m1 = fmaxf(m1, c);
}
// 16-bit heads: exact ties of the largest logit are common (bfloat16 keeps 8 significant bits: ~1.5 % of dense
// candidates), and with the update above every tie takes the literal re-evaluation (80 scattered re-reads), which halved
// the bfloat16 throughput.  Here m2 is the largest value STRICTLY below m1 and k0 the lowest index holding m1 in any
// visiting order.  Same result: when m2 < guard_lo every class value in the guard band equals m1, so the literal path
// would score exactly those classes, all alike, and keep the lowest index -- k0, with score and smax of the fast path.
// Distinct values inside the band still take the literal path.
template <typename T>
__device__ __forceinline__ void top2_update_t(float c, int k, float &m1, float &m2, int &k0)
{
    if (sizeof(T) == 4) {
        top2_update(c, k, m1, m2, k0);
        return;
    }
    m2 = (c < m1) ? fmaxf(m2, c) : ((c > m1) ? m1 : m2);
    k0 = (c > m1 || (c == m1 && k < k0)) ? k : k0;
    m1 = fmaxf(m1, c);
}

// Decide one candidate.  m1/m2/k0: largest, second largest class value and first index of the largest; objv:
// objectness logit (or probability when DECODED); read_cls(k) re-reads class value k (slow path only).
// Returns true when the candidate survives; pre_pass reports the pre-mask (FCOS top-k needs its count).
template <bool DECODED, class ReadCls>
__device__ __forceinline__ bool decide_candidate(const Plan &P, float m1, float m2, int k0, float objv,
                                                 ReadCls read_cls, float &score, int &cls, bool &pre_pass)
{
    pre_pass = false;
    const float mult = P.use_obj ? (DECODED ? objv : sigmoid_ref(objv)) : 1.0f;
    if (P.pre_kind == PRE_OBJ && !(mult >= P.conf_thr)) return false;
    float smax, p, guard_lo;
    if (DECODED) {
        smax = m1;
        p = P.use_obj ? __fmul_rn(m1, mult) : m1;
        guard_lo = __fmul_rn(m1, 1.0f - 2.0e-6f);  // products of values this close may round together
        if (!(m1 > 0.0f) || !(p > 1.0e-30f)) guard_lo = -INFINITY;
    } else {
        const float e = expf(-m1);
        smax = __fdiv_rn(1.0f, __fadd_rn(1.0f, e));
        p = P.use_obj ? __fmul_rn(smax, mult) : smax;
        // d/dx ln sigmoid(x) = sigmoid(-x) >= sigmoid(-m1) on [m1-d, m1]: a logit gap d = 8e-6 * (1 + e^m1)
        // guarantees a relative sigmoid gap > 4e-6, far above the <= 1e-6 the implementation can blur.
        guard_lo = m1 - 8.0e-6f * (1.0f + __fdiv_rn(1.0f, e));
        if (m1 < -80.0f || !(p > 1.0e-30f) || !(guard_lo == guard_lo)) guard_lo = -INFINITY;
    }
    cls = k0;
    if (!(m2 < guard_lo)) {
        // near-tie (or denormal range): literal evaluation of every class that could reach the maximum.  Values are
        // re-read 8 at a time with independent loads (a load-per-iteration loop would serialise 80 DRAM round trips
        // and stall the whole warp for tens of microseconds).
        float best = -INFINITY;
        int kb = 0;
        float sbest = -INFINITY;
        for (int kc = 0; kc < P.C; kc += 8) {
            float cv[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) cv[j] = (kc + j < P.C) ? read_cls(kc + j) : -INFINITY;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const float c = cv[j];
                if (kc + j < P.C && c >= guard_lo) {
                    const float sk = DECODED ? c : sigmoid_ref(c);
                    const float pk = P.use_obj ? __fmul_rn(sk, mult) : sk;
                    if (pk > best) { best = pk; kb = kc + j; }
                    sbest = fmaxf(sbest, sk);
                }
            }
        }
        p = best;
        cls = kb;
        smax = sbest;
    }
    switch (P.pre_kind) {
    case PRE_OBJ_X_MAX: pre_pass = p >= P.conf_thr; break;  // fl(obj * max cls) == max fl(obj * cls)
    case PRE_MAXCLS: pre_pass = smax >= P.cls_thr; break;
    case PRE_ANY_GT: pre_pass = smax > P.pre_thr; break;
    default: pre_pass = true; break;
    }
    if (!pre_pass) return false;
    score = p;
    return P.post_strict ? (p > P.cls_thr) : (p >= P.cls_thr);
}

// Warp-aggregated append of up to VEC keys per thread (okm: bit j set when k[j] is a survivor).
// ext_seen: the image's running score extrema (cnt[2], cnt[3]) as read EARLIER by the caller (kernel start: the load's
// latency hides behind the scan; a stale value only means a redundant fire-and-forget atomicMax), or nullptr: read here,
// issued before the slot reservation so that the two round trips overlap instead of adding up.
template <int VEC>
__device__ __forceinline__ void emit_keys(const uint64_t (&k)[VEC], unsigned okm, int npre, uint32_t smax_bits,
                                          uint32_t smin_inv, uint64_t *keys_img, int64_t cap, int32_t *cnt, bool count_pre,
                                          const uint2 *ext_seen = nullptr)
{
    const unsigned lane = threadIdx.x & 31u;
    const int nk = __popc(okm);
    int incl = nk;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const int v = __shfl_up_sync(0xffffffffu, incl, d);
        if (lane >= static_cast<unsigned>(d)) incl += v;
    }
    const int total = __shfl_sync(0xffffffffu, incl, 31);
    if (count_pre) {
        const int tp = __reduce_add_sync(0xffffffffu, npre);
        if (lane == 0 && tp) atomicAdd(cnt + 1, tp);
    }
    if (total == 0) return;
    const uint32_t wmax = __reduce_max_sync(0xffffffffu, smax_bits);
    const uint32_t wmin = __reduce_max_sync(0xffffffffu, smin_inv);
    int base = 0;
    if (lane == 0) {
        // the running extrema rarely change after the first warps of an image: look before touching them
        uint2 ext;
        if (ext_seen) {
            ext = *ext_seen;
        } else {
            const volatile unsigned int *e = reinterpret_cast<const volatile unsigned int *>(cnt + 2);
            ext.x = e[0];
            ext.y = e[1];
        }
        base = atomicAdd(cnt, total);
        if (wmax > ext.x) atomicMax(reinterpret_cast<unsigned int *>(cnt + 2), wmax);
        if (wmin > ext.y) atomicMax(reinterpret_cast<unsigned int *>(cnt + 3), wmin);
    }
    base = __shfl_sync(0xffffffffu, base, 0);
    const int64_t at = static_cast<int64_t>(base) + (incl - nk);
#pragma unroll
    for (int j = 0; j < VEC; ++j) {
        const int64_t slot = at + __popc(okm & ((1u << j) - 1u));
        if (((okm >> j) & 1u) && slot < cap) keys_img[slot] = k[j];
    }
}

// -------------------------------------------------------------------------------------------------------
// planes layout (NCHW heads: YOLOv5, YOLOX, YOLOv8, FCOS).  One thread = VEC consecutive positions of one
// (image, anchor); per class plane a warp reads 32*VEC*4 contiguous bytes (512 B with 128-bit loads).
// -------------------------------------------------------------------------------------------------------
template <typename T, int VEC, int U = 8, int THREADS = 256, int MINB = 1, int HINT = 0, int PROBE = 0, bool WIDE = false>
__global__ void __launch_bounds__(THREADS, MINB) k_filter_planes(const __grid_constant__ Plan P, uint64_t *__restrict__ keys,
                                                                 int64_t key_cap, int32_t *__restrict__ counts)
{
    // blockIdx.x = image: CTAs that run at the same time append to DIFFERENT images' counters (the per-image
    // atomicAdd is the only contended address of the kernel)
    const bool img_fast = gridDim.x == static_cast<unsigned>(P.batch) && gridDim.y != static_cast<unsigned>(P.batch);
    const int img = img_fast ? blockIdx.x : blockIdx.y;
    const int u = (img_fast ? blockIdx.y : blockIdx.x) * blockDim.x + threadIdx.x;
    const bool active = u < P.units_per_img;
    uint64_t out[VEC];
    unsigned okm = 0u;
    int npre = 0;
    uint32_t smax_bits = 0u, smin_inv = 0u;
#pragma unroll
    for (int j = 0; j < VEC; ++j) out[j] = 0ull;
    if (active) {
        int l = 0;
#pragma unroll
        for (int i = 1; i < YSB_MAX_LEVELS; ++i)
            if (i < P.L && u >= P.lv[i].unit_off) l = i;
        const LevelDesc &lv = P.lv[l];
        const bool vec4 = VEC == 4 && lv.vec == 4;  // levels whose planes are not 4-element sized use one position per unit
        const int upos = vec4 ? 4 : 1;
        const int upa = lv.hw / upos;  // units per anchor
        const int ru = u - lv.unit_off;
        const int a = ru / upa;
        const int pos = (ru - a * upa) * upos;
        const int cand0 = lv.cand_off + a * lv.hw + pos;
        const size_t hw = static_cast<size_t>(lv.hw);
        const T *cls = head_ptr<T>(lv.p0) + (static_cast<size_t>(img * P.A + a) * P.cls_nch + P.cls_ch) * hw + pos;

        float m1[VEC], m2[VEC];
        int k0[VEC];
#pragma unroll
        for (int j = 0; j < VEC; ++j) { m1[j] = -INFINITY; m2[j] = -INFINITY; k0[j] = 0; }

        // U independent 128-bit loads in flight per thread
        int k = 0;
        for (; k + U <= P.C; k += U) {
            float v[U][VEC];
#pragma unroll
            for (int q = 0; q < U; ++q) {
                if (vec4) {
                    const float4 t = HINT ? ldg_stream4_256(cls + static_cast<size_t>(k + q) * hw) : ldg_stream4(cls + static_cast<size_t>(k + q) * hw);
                    v[q][0] = t.x; v[q][1 % VEC] = t.y; v[q][2 % VEC] = t.z; v[q][3 % VEC] = t.w;
                } else {
                    v[q][0] = ldg_stream1(cls + static_cast<size_t>(k + q) * hw);
#pragma unroll
                    for (int j = 1; j < VEC; ++j) v[q][j] = -INFINITY;
                }
            }
#pragma unroll
            for (int q = 0; q < U; ++q)
#pragma unroll
                for (int j = 0; j < VEC; ++j) {
                    if (PROBE) m1[j] = fmaxf(m1[j], v[q][j]);  // profiling aid: same loads, 1 ALU op per logit
                    else top2_update_t<T>(v[q][j], k + q, m1[j], m2[j], k0[j]);
                }
        }
        for (; k < P.C; ++k) {
            float v[VEC];
            if (vec4) {
                const float4 t = ldg_stream4(cls + static_cast<size_t>(k) * hw);
                v[0] = t.x; v[1 % VEC] = t.y; v[2 % VEC] = t.z; v[3 % VEC] = t.w;
            } else {
                v[0] = ldg_stream1(cls + static_cast<size_t>(k) * hw);
#pragma unroll
                for (int j = 1; j < VEC; ++j) v[j] = -INFINITY;
            }
#pragma unroll
            for (int j = 0; j < VEC; ++j) top2_update_t<T>(v[j], k, m1[j], m2[j], k0[j]);
        }
        float objv[VEC];
#pragma unroll
        for (int j = 0; j < VEC; ++j) objv[j] = 0.0f;
        if (P.use_obj) {
            const T *ob = head_ptr<T>(P.obj_src == 2 ? lv.p2 : lv.p0) +
                          (static_cast<size_t>(img * P.A + a) * P.obj_nch + P.obj_ch) * hw + pos;
            if (vec4) {
                const float4 t = ldg_stream4(ob);
                objv[0] = t.x; objv[1 % VEC] = t.y; objv[2 % VEC] = t.z; objv[3 % VEC] = t.w;
            } else {
                objv[0] = ldg_stream1(ob);
            }
        }
#pragma unroll
        for (int j = 0; j < VEC; ++j) {
            if (j >= upos) break;
            float score;
            int c;
            bool pre;
            const T *cj = cls + j;
            const bool ok = decide_candidate<false>(
                P, m1[j], m2[j], k0[j], objv[j], [&](int kk) { return ldg_head(cj + static_cast<size_t>(kk) * hw); },
                score, c, pre);
            npre += pre ? 1 : 0;
            if (ok) {
                out[j] = pack_key<WIDE>(score, static_cast<uint32_t>(P.cand_base + cand0 + j), static_cast<uint32_t>(c));
                okm |= 1u << j;
                const uint32_t sb = __float_as_uint(score);
                smax_bits = max(smax_bits, sb);
                smin_inv = max(smin_inv, ~sb);
            }
        }
    }
    emit_keys<VEC>(out, okm, npre, smax_bits, smin_inv, keys + static_cast<int64_t>(img) * key_cap, key_cap,
                   counts + img * 4, P.pre_kind == PRE_ANY_GT);
}
// -------------------------------------------------------------------------------------------------------
// planes layout, every level 128-bit loadable (the common case: H*W % 4 == 0 on all levels, 16-byte aligned heads).
// Same decomposition and results as k_filter_planes<4>; specialised so that
//   * there is no per-level scalar fallback path (the generic kernel if-converts both paths and issues both),
//   * plane addresses are 32-bit element offsets from the (image, anchor) block (2 integer ops per load instead of 6),
//   * the last C % U class planes and the objectness plane are ONE batch of independent loads (the generic kernel walks
//     the remainder one dependent load at a time and fetches objectness after the whole class scan).
// -------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void prefetch_l2(const void *p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }

// PF > 0: while the loads of batch b are in flight, the lines of batch b + PF are requested into L2 with prefetch
// instructions (no registers held): the demand loads of later batches then hit L2 instead of waiting a DRAM round trip.
template <typename T, int U, int THREADS, int MINB, int PF = 0, bool WIDE = false>
__global__ void __launch_bounds__(THREADS, MINB) k_filter_planes_v4(const __grid_constant__ Plan P, uint64_t *__restrict__ keys,
                                                                    int64_t key_cap, int32_t *__restrict__ counts)
{
    const int img = blockIdx.x;  // image-fastest grid: concurrent CTAs append to different per-image counters
    const int u = blockIdx.y * THREADS + threadIdx.x;
    const bool active = u < P.units_per_img;
    uint64_t out[4] = {0ull, 0ull, 0ull, 0ull};
    unsigned okm = 0u;
    int npre = 0;
    uint32_t smax_bits = 0u, smin_inv = 0u;
    if (active) {
        int l = 0;
#pragma unroll
        for (int i = 1; i < YSB_MAX_LEVELS; ++i)
            if (i < P.L && u >= P.lv[i].unit_off) l = i;
        const LevelDesc &lv = P.lv[l];
        const uint32_t hw = static_cast<uint32_t>(lv.hw);
        const int upa = lv.hw >> 2;  // units per anchor
        const int ru = u - lv.unit_off;
        const int a = ru / upa;
        const int pos = (ru - a * upa) << 2;
        const int cand0 = lv.cand_off + a * lv.hw + pos;
        const T *cls = head_ptr<T>(lv.p0) + (static_cast<size_t>(img * P.A + a) * P.cls_nch + P.cls_ch) * hw + pos;
        const int C = P.C;

        float m1[4], m2[4], objv[4];
        int k0[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) { m1[j] = -INFINITY; m2[j] = -INFINITY; k0[j] = 0; objv[j] = 0.0f; }

        int k = 0;
        uint32_t off = 0;  // k * hw, in elements: an (image, anchor) block is far below 2^32 elements
        if (PF > 0 && (threadIdx.x & 7) == 0) {
            // prime the pipeline: batches 1 .. PF (8 lanes share a 128-byte line; one of them asks for it)
#pragma unroll
            for (int q = 0; q < PF * U; ++q)
                if (U + q < C) prefetch_l2(cls + (U + q) * hw);
        }
        for (; k + U <= C; k += U, off += U * hw) {
            float4 v[U];
#pragma unroll
            for (int q = 0; q < U; ++q) v[q] = ldg_stream4_256(cls + (off + q * hw));
            if (PF > 0 && (threadIdx.x & 7) == 0) {
#pragma unroll
                for (int q = 0; q < U; ++q) {
                    const int kk = k + (PF + 1) * U + q;
                    if (kk < C) prefetch_l2(cls + (off + ((PF + 1) * U + q) * hw));
                }
                if (P.use_obj && k == 0)
                    prefetch_l2(head_ptr<T>(P.obj_src == 2 ? lv.p2 : lv.p0) + (static_cast<size_t>(img * P.A + a) * P.obj_nch + P.obj_ch) * hw + pos);
            }
#pragma unroll
            for (int q = 0; q < U; ++q) {
                top2_update_t<T>(v[q].x, k + q, m1[0], m2[0], k0[0]);
                top2_update_t<T>(v[q].y, k + q, m1[1], m2[1], k0[1]);
                top2_update_t<T>(v[q].z, k + q, m1[2], m2[2], k0[2]);
                top2_update_t<T>(v[q].w, k + q, m1[3], m2[3], k0[3]);
            }
        }
        {
            // tail batch: the remaining (< U) class planes and the objectness plane, all in flight together
            const int rem = C - k;
            float4 v[U];
            float4 ov = make_float4(0.f, 0.f, 0.f, 0.f);
            if (P.use_obj) {
                const T *ob = head_ptr<T>(P.obj_src == 2 ? lv.p2 : lv.p0) +
                              (static_cast<size_t>(img * P.A + a) * P.obj_nch + P.obj_ch) * hw + pos;
                ov = ldg_stream4_256(ob);
            }
#pragma unroll
            for (int q = 0; q < U - 1; ++q)
                if (q < rem) v[q] = ldg_stream4_256(cls + (off + q * hw));
#pragma unroll
            for (int q = 0; q < U - 1; ++q)
                if (q < rem) {
                    top2_update_t<T>(v[q].x, k + q, m1[0], m2[0], k0[0]);
                    top2_update_t<T>(v[q].y, k + q, m1[1], m2[1], k0[1]);
                    top2_update_t<T>(v[q].z, k + q, m1[2], m2[2], k0[2]);
                    top2_update_t<T>(v[q].w, k + q, m1[3], m2[3], k0[3]);
                }
            objv[0] = ov.x; objv[1] = ov.y; objv[2] = ov.z; objv[3] = ov.w;
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            float score;
            int c;
            bool pre;
            const T *cj = cls + j;
            const bool ok = decide_candidate<false>(
                P, m1[j], m2[j], k0[j], objv[j], [&](int kk) { return ldg_head(cj + static_cast<size_t>(kk) * hw); }, score, c, pre);
            npre += pre ? 1 : 0;
            if (ok) {
                out[j] = pack_key<WIDE>(score, static_cast<uint32_t>(P.cand_base + cand0 + j), static_cast<uint32_t>(c));
                okm |= 1u << j;
                const uint32_t sb = __float_as_uint(score);
                smax_bits = max(smax_bits, sb);
                smin_inv = max(smin_inv, ~sb);
            }
        }
    }
    emit_keys<4>(out, okm, npre, smax_bits, smin_inv, keys + static_cast<int64_t>(img) * key_cap, key_cap, counts + img * 4,
                 P.pre_kind == PRE_ANY_GT);
}

// shared-memory staging helpers (k_filter_rows; the profiling variants)
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }
__device__ __forceinline__ void cp_async16(uint32_t dst_smem, const void *src)
{
    asm volatile("cp.async.cg.shared.global.L2::128B [%0], [%1], 16;" ::"r"(dst_smem), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait()
{
    asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory");
}

// mbarrier + bulk-copy (TMA engine) helpers
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity)
{
    asm volatile(
        "{\n"
        ".reg .pred P1;\n"
        "LAB_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
        "@P1 bra DONE;\n"
        "bra LAB_WAIT;\n"
        "DONE:\n"
        "}\n" ::"r"(bar),
        "r"(parity)
        : "memory");
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst_smem, const void *src_gmem, uint32_t bytes, uint32_t bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst_smem),
                 "l"(src_gmem), "r"(bytes), "r"(bar)
                 : "memory");
}

#ifdef YSB_PROFILING_VARIANTS
#include "filter_variants.cuh"
#endif

// -------------------------------------------------------------------------------------------------------
// rows layout (channels-last heads: YOLOv7, RetinaNet cls, NHWC YOLOv5 / YOLOX / YOLOv8 / FCOS cls; and the decoded
// (b, N, C') tensor of any family).
// A CTA stages a tile of 128 whole rows in shared memory with one bulk copy (rows are 340 B / 320 B and only 4-byte
// aligned individually, but the tile is contiguous and 16-byte aligned), then one thread scans one row: 128-bit shared
// loads when the class run of every row is 16-byte aligned, else scalar loads; rows with an even stride are walked with
// a per-thread rotation so that the rows a warp scans sit in different banks.
// 16-bit heads are staged as they are (rows of 170 B / 160 B, 2-byte aligned) and widened as the scan reads them.  The
// copy engines move 16-byte multiples from 16-byte aligned addresses, so a tile takes the bulk path when its first
// element is 16-byte aligned and its length is a multiple of 16 bytes (8 elements here, 4 for float32): true for every
// full tile of both layouts (128 rows x 170 B = 1360 x 16 B) and for every tail at a 640x640 input;
// anything else is staged with scalar loads.
// -------------------------------------------------------------------------------------------------------
constexpr int kRowsTile = 128;

// One thread scans one staged row (thread t of the tile -> row r0 + t of level lv), decides it and the warp appends the
// survivors.  Every thread of the warp must call (rows beyond nrows contribute nothing).
// NHWC: the tile holds rows of channels-last planes-family heads (YOLOv5, YOLOX, YOLOv8, FCOS cls): memory row m of a level
// is candidate a*hw + p with p = m / A, a = m % A, and FCOS' centerness is read from its own (b, H, W, 1) tensor.
template <typename T, bool NHWC = false>
__device__ __forceinline__ void rows_scan_emit(const Plan &P, const LevelDesc &lv, int img, const T *tile, int sstride,
                                               int nrows, int r0, int t, uint64_t *__restrict__ keys, int64_t key_cap,
                                               int32_t *__restrict__ counts, bool vec4 = false, const uint2 *ext_seen = nullptr)
{
    uint64_t out[1] = {0ull};
    unsigned okm = 0u;
    int npre = 0;
    uint32_t smax_bits = 0u, smin_inv = 0u;
    if (t < nrows) {
        const T *row = tile + t * sstride;
        const T *cls = row + P.cls_col_in;
        float m1 = -INFINITY, m2 = -INFINITY;
        int k0 = 0;
        // thread t reads word sstride*t + k: conflict-free when sstride is odd; otherwise start the walk at column t so
        // that the 32 lanes hit (sstride+1)*t + k.  The visiting order is irrelevant: a unique maximum has a unique
        // index, and equal maxima force m2 == m1, i.e. the literal path, which walks in index order.
        if (sizeof(T) == 4 && vec4 && ((sstride | P.cls_col_in | P.C) & 3) == 0) {
            // 16-byte aligned class runs (RetinaNet's 80-float rows, 84-float decoded rows): 128-bit shared loads, four
            // independent (max, runner-up, position) chains -- one per float4 component -- that share the float4's
            // position, merged at the end.  A quarter-warp reads 8 float4 per wavefront: with an even number of float4 per
            // row the lanes start at float4 `lane & 7` (8 consecutive rows then sit in 8 different 16-byte bank groups), with an
            // odd number the straight walk already is conflict-free.  Visiting order and chain split cannot change the
            // result: a unique maximum has one position, and equal maxima -- within a chain or across chains -- surface
            // as runner-up == maximum, i.e. the literal path below.
            const int nq = P.C >> 2, R = sstride >> 2;
            const float4 *c4 = reinterpret_cast<const float4 *>(cls);
            float a1[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY}, a2[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};
            int aq[4] = {0, 0, 0, 0};
            int q = (R & 1) ? 0 : (t & 7) % nq;   // 128-bit loads are served a quarter-warp at a time
#pragma unroll 4
            for (int s = 0; s < nq; ++s) {
                const float4 v = c4[q];
                const float c[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    a2[j] = fmaxf(a2[j], fminf(a1[j], c[j]));
                    aq[j] = (c[j] > a1[j]) ? q : aq[j];
                    a1[j] = fmaxf(a1[j], c[j]);
                }
                if (++q == nq) q = 0;
            }
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                m2 = fmaxf(fmaxf(m2, a2[j]), fminf(m1, a1[j]));
                k0 = (a1[j] > m1) ? 4 * aq[j] + j : k0;
                m1 = fmaxf(m1, a1[j]);
            }
        } else if (sstride & 1) {
            // odd stride (YOLOv7's 85-float rows): already conflict-free, a straight run without the wrap test
#pragma unroll 8
            for (int k = 0; k < P.C; ++k) top2_update_t<T>(widen(cls[k]), k, m1, m2, k0);
        } else {
            // rotated walk: lane l starts at column l, i.e. reads word sstride*tid + l + t = (sstride + 1)*l + t (mod 32)
            // -- an odd multiplier, conflict-free.  Every lane runs the same C iterations (two straight runs per lane
            // would diverge); the first C - 32 of them cannot wrap, so only the last 32 carry the wrap test.
            const int lane = t & 31;
            if (P.C >= 32) {
                const int straight = P.C - 32;
#pragma unroll 8
                for (int t = 0; t < straight; ++t) top2_update_t<T>(widen(cls[t + lane]), t + lane, m1, m2, k0);
                int k = straight + lane;
#pragma unroll 8
                for (int t = 0; t < 32; ++t) {
                    if (k >= P.C) k -= P.C;
                    top2_update_t<T>(widen(cls[k]), k, m1, m2, k0);
                    ++k;
                }
            } else {
                int k = lane % P.C;
                for (int t = 0; t < P.C; ++t) {
                    top2_update_t<T>(widen(cls[k]), k, m1, m2, k0);
                    if (++k == P.C) k = 0;
                }
            }
        }
        int cand = lv.cand_off + r0 + t, pos = 0;
        if (NHWC) {
            const int m = r0 + t, a = m % P.A;
            pos = m / P.A;
            cand = lv.cand_off + a * lv.hw + pos;
        }
        float objv = 0.0f;
        if (P.use_obj) {
            if (NHWC && P.obj_src == 2)  // FCOS centerness (A == 1)
                objv = ldg_head(head_elem<T, true>(lv, lv.p2, 1, P.obj_nch, img, 0, pos, P.obj_ch));
            else if (P.obj_src == 1)  // RetinaNet-exp: conf logit is the last column of the reg tensor
                objv = ldg_head(head_ptr<T>(P.lv[0].p1) + (static_cast<size_t>(img) * P.N + cand) * P.reg_row_w + 4);
            else
                objv = widen(row[P.obj_col_in]);
        }
        float score;
        int c;
        bool pre, ok;
        if (P.input_kind == YSB_INPUT_DECODED_ROWS)
            ok = decide_candidate<true>(P, m1, m2, k0, objv, [&](int kk) { return widen(cls[kk]); }, score, c, pre);
        else
            ok = decide_candidate<false>(P, m1, m2, k0, objv, [&](int kk) { return widen(cls[kk]); }, score, c, pre);
        npre = pre ? 1 : 0;
        if (ok) {
            out[0] = pack_key(score, static_cast<uint32_t>(P.cand_base + cand), static_cast<uint32_t>(c));
            okm = 1u;
            smax_bits = __float_as_uint(score);
            smin_inv = ~smax_bits;
        }
    }
    emit_keys<1>(out, okm, npre, smax_bits, smin_inv, keys + static_cast<int64_t>(img) * key_cap, key_cap,
                 counts + img * 4, P.pre_kind == PRE_ANY_GT, ext_seen);
}

template <typename T, bool NHWC>
__global__ void __launch_bounds__(kRowsTile) k_filter_rows(const __grid_constant__ Plan P, uint64_t *__restrict__ keys,
                                                           int64_t key_cap, int32_t *__restrict__ counts, int flags)
{
    extern __shared__ __align__(128) float tile_f[];
    T *tile = reinterpret_cast<T *>(tile_f);
    constexpr int kVecShift = sizeof(T) == 4 ? 2 : 3;   // log2 of the elements in 16 bytes
    const int img = blockIdx.x;  // image fastest: see k_filter_planes
    const int t = blockIdx.y;
    int l = 0;
#pragma unroll
    for (int i = 1; i < YSB_MAX_LEVELS; ++i)
        if (i < P.L && t >= P.lv[i].unit_off) l = i;
    const LevelDesc &lv = P.lv[l];
    const int rows_l = (l + 1 < P.L ? P.lv[l + 1].cand_off : P.N) - lv.cand_off;
    const int r0 = (t - lv.unit_off) * kRowsTile;
    const int nrows = min(kRowsTile, rows_l - r0);
    const int rw = P.row_w_in;
    const T *src = head_ptr<T>(lv.p0) + (static_cast<size_t>(img) * lv.img_rows + r0) * rw;
    const int nfl = nrows * rw;
    // the image's running score extrema, read now so that the load hides behind the staging copy (see emit_keys)
    const volatile unsigned int *ext_p = reinterpret_cast<const volatile unsigned int *>(counts + img * 4 + 2);
    const uint2 ext_seen = make_uint2(ext_p[0], ext_p[1]);
    // 16-byte aligned tiles (every reference layout): cp.async straight into a DENSE shared tile -- no register
    // staging, no per-element address math.  Rows with an even float stride are scanned with a per-thread rotation
    // (below) instead of padding.  Odd shapes: scalar loads into a tile padded to an odd stride.
    const bool dense = ((reinterpret_cast<uintptr_t>(src) & 15u) == 0) && ((nfl & ((1 << kVecShift) - 1)) == 0);
    const int sstride = dense ? rw : (rw | 1);
    if (dense && !(flags & 1)) {
        const uint32_t dst = smem_u32(tile);
        const int nv = nfl >> kVecShift;
        for (int i = threadIdx.x; i < nv; i += kRowsTile) cp_async16(dst + 16u * i, src + (1 << kVecShift) * i);
        cp_async_commit();
        cp_async_wait<0>();
    } else if (dense) {
        // the tile is one contiguous block: ONE bulk copy of the TMA engine (cp.async.bulk -> mbarrier complete_tx) issued
        // by thread 0 instead of 20 cp.async per thread
        __shared__ __align__(8) uint64_t bar;
        const uint32_t b32 = smem_u32(&bar);
        if (threadIdx.x == 0) {
            mbar_init(b32, 1);
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
            mbar_expect_tx(b32, static_cast<uint32_t>(nfl) * static_cast<uint32_t>(sizeof(T)));
            bulk_g2s(smem_u32(tile), src, static_cast<uint32_t>(nfl) * static_cast<uint32_t>(sizeof(T)), b32);
        }
        __syncthreads();   // the barrier is initialised before anybody polls it
        mbar_wait(b32, 0u);
    } else {
        for (int e = threadIdx.x; e < nfl; e += kRowsTile) {
            const int row = e / rw, col = e - row * rw;
            tile[row * sstride + col] = ldg_stream1_raw(src + e);
        }
    }
    __syncthreads();

    rows_scan_emit<T, NHWC>(P, lv, img, tile, sstride, nrows, r0, static_cast<int>(threadIdx.x), keys, key_cap, counts,
                            (flags & 2) != 0, &ext_seen);
}

// -------------------------------------------------------------------------------------------------------
// rows layout, rows wider than the 128-row shared tile (!rows_fit_tile: YOLOv7 rows of 5 + C from C = 449, RetinaNet /
// RetinaNet-exp class rows from C = 454, decoded rows; up to 2048 classes, narrow or wide keys).
// Same grid as k_filter_rows (one CTA per image and 128-row tile), no shared memory: warp w scans rows 32w .. 32w + 31 of
// the tile one at a time, the whole warp on one row, straight from global memory in 16-byte loads (4 float32 / 8 16-bit
// values; a row start that is not 16-byte aligned -- YOLOv7's 5 + C values -- is peeled into scalar head and tail loads).
// Each lane keeps its own (max, runner-up, first index of max) over the columns it visits in ascending order; the lanes
// merge by butterfly shuffle (merge_top2), and lane j keeps row 32w + j.  Then every lane decides its row with the tail
// of rows_scan_emit (decide_candidate, whose literal path re-reads the row from global memory) and the warp appends.
// -------------------------------------------------------------------------------------------------------
constexpr int kWideRowsInFlight = 4;   // 16-byte loads in flight per lane

__device__ __forceinline__ void ldg16(const float *p, float (&v)[4])
{
    const float4 t = ldg_stream4(p);
    v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
}
template <typename T>
__device__ __forceinline__ void ldg16(const T *p, float (&v)[8])
{
    uint4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
    const float4 a = widen4(make_uint2(r.x, r.y), p), b = widen4(make_uint2(r.z, r.w), p);
    v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
}

// Merge another lane's (b1, b2, bk) into (m1, m2, k0), with the semantics of top2_update_t<T>: float32 -- equal maxima
// leave runner-up == maximum (the literal path); 16-bit -- m2 is the largest value strictly below m1 and k0 the lowest
// index of m1.  Symmetric, so every lane of a butterfly ends with the same triple.
template <typename T>
__device__ __forceinline__ void merge_top2(float &m1, float &m2, int &k0, float b1, float b2, int bk)
{
    if (sizeof(T) == 4) m2 = fmaxf(fmaxf(m2, b2), fminf(m1, b1));
    else m2 = (b1 > m1) ? fmaxf(m1, b2) : ((b1 < m1) ? fmaxf(m2, b1) : fmaxf(m2, b2));
    k0 = (b1 > m1 || (b1 == m1 && bk < k0)) ? bk : k0;
    m1 = fmaxf(m1, b1);
}

template <typename T, bool WIDE>
__global__ void __launch_bounds__(kRowsTile) k_filter_rows_wide(const __grid_constant__ Plan P, uint64_t *__restrict__ keys,
                                                                int64_t key_cap, int32_t *__restrict__ counts)
{
    constexpr int E = 16 / static_cast<int>(sizeof(T));   // values per 16-byte load
    const int img = blockIdx.x;
    const int t = blockIdx.y;
    int l = 0;
#pragma unroll
    for (int i = 1; i < YSB_MAX_LEVELS; ++i)
        if (i < P.L && t >= P.lv[i].unit_off) l = i;
    const LevelDesc &lv = P.lv[l];
    const int rows_l = (l + 1 < P.L ? P.lv[l + 1].cand_off : P.N) - lv.cand_off;
    const int r0 = (t - lv.unit_off) * kRowsTile;
    const int nrows = min(kRowsTile, rows_l - r0);
    const int rw = P.row_w_in, C = P.C;
    const T *tile = head_ptr<T>(lv.p0) + (static_cast<size_t>(img) * lv.img_rows + r0) * rw;
    const volatile unsigned int *ext_p = reinterpret_cast<const volatile unsigned int *>(counts + img * 4 + 2);
    const uint2 ext_seen = make_uint2(ext_p[0], ext_p[1]);
    const int lane = threadIdx.x & 31;
    const int wr0 = (threadIdx.x >> 5) * 32;

    float my1 = -INFINITY, my2 = -INFINITY;
    int myk = 0;
    for (int i = 0; i < 32 && wr0 + i < nrows; ++i) {   // warp-uniform
        const T *cls = tile + static_cast<size_t>(wr0 + i) * rw + P.cls_col_in;
        const int head = min(C, static_cast<int>(((16u - (reinterpret_cast<uintptr_t>(cls) & 15u)) & 15u) / sizeof(T)));
        const int nv = (C - head) / E;
        const int tail0 = head + nv * E;
        float m1 = -INFINITY, m2 = -INFINITY;
        int k0 = 0;
        if (lane < head) top2_update_t<T>(ldg_stream1(cls + lane), lane, m1, m2, k0);
        const T *body = cls + head;
        for (int v0 = 0; v0 < nv; v0 += 32 * kWideRowsInFlight) {
            float x[kWideRowsInFlight][E];
#pragma unroll
            for (int q = 0; q < kWideRowsInFlight; ++q) {
                const int v = v0 + 32 * q + lane;
                if (v < nv) {
                    ldg16(body + static_cast<size_t>(v) * E, x[q]);
                } else {
#pragma unroll
                    for (int j = 0; j < E; ++j) x[q][j] = -INFINITY;
                }
            }
#pragma unroll
            for (int q = 0; q < kWideRowsInFlight; ++q) {
                const int k = head + (v0 + 32 * q + lane) * E;
#pragma unroll
                for (int j = 0; j < E; ++j) top2_update_t<T>(x[q][j], k + j, m1, m2, k0);
            }
        }
        if (tail0 + lane < C) top2_update_t<T>(ldg_stream1(cls + tail0 + lane), tail0 + lane, m1, m2, k0);
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) {
            const float b1 = __shfl_xor_sync(0xffffffffu, m1, d), b2 = __shfl_xor_sync(0xffffffffu, m2, d);
            const int bk = __shfl_xor_sync(0xffffffffu, k0, d);
            merge_top2<T>(m1, m2, k0, b1, b2, bk);
        }
        if (lane == i) { my1 = m1; my2 = m2; myk = k0; }
    }

    uint64_t out[1] = {0ull};
    unsigned okm = 0u;
    int npre = 0;
    uint32_t smax_bits = 0u, smin_inv = 0u;
    const int rj = wr0 + lane;
    if (rj < nrows) {
        const T *row = tile + static_cast<size_t>(rj) * rw;
        const T *cls = row + P.cls_col_in;
        const int cand = lv.cand_off + r0 + rj;
        float objv = 0.0f;
        if (P.use_obj)
            objv = P.obj_src == 1 ? ldg_head(head_ptr<T>(P.lv[0].p1) + (static_cast<size_t>(img) * P.N + cand) * P.reg_row_w + 4)
                                  : ldg_head(row + P.obj_col_in);
        float score;
        int c;
        bool pre, ok;
        if (P.input_kind == YSB_INPUT_DECODED_ROWS)
            ok = decide_candidate<true>(P, my1, my2, myk, objv, [&](int kk) { return ldg_head(cls + kk); }, score, c, pre);
        else
            ok = decide_candidate<false>(P, my1, my2, myk, objv, [&](int kk) { return ldg_head(cls + kk); }, score, c, pre);
        npre = pre ? 1 : 0;
        if (ok) {
            out[0] = pack_key<WIDE>(score, static_cast<uint32_t>(P.cand_base + cand), static_cast<uint32_t>(c));
            okm = 1u;
            smax_bits = __float_as_uint(score);
            smin_inv = ~smax_bits;
        }
    }
    emit_keys<1>(out, okm, npre, smax_bits, smin_inv, keys + static_cast<int64_t>(img) * key_cap, key_cap, counts + img * 4,
                 P.pre_kind == PRE_ANY_GT, &ext_seen);
}

#ifdef YSB_PROFILING_VARIANTS
// -------------------------------------------------------------------------------------------------------
// rows layout, persistent ring version (profiling build, YSB_ROWS_RING=1; measured SLOWER than k_filter_rows: 8 scanning
// warps per SM cannot hide the shared-memory latency of the top-2 scan -- RetinaNet b=64 0.447 vs 0.324 ms).
// A tile of 128 rows is ONE contiguous block of memory (40-44 KB), i.e. one bulk copy of the TMA engine
// (cp.async.bulk -> mbarrier complete_tx): a CTA keeps kRingStages tiles in flight / under the scan, thread 0 re-arms a
// stage as soon as the CTA has finished reading it.  Against k_filter_rows (one tile per CTA: ~300 CTA launches per SM
// for a RetinaNet batch, 20 cp.async per thread and tile, no copy/scan overlap inside a CTA) this removes the per-tile
// CTA turnaround and the load-issue instructions.  Work item w -> (image w % batch, unit w / batch): image fastest, so
// CTAs that run at the same time append to different images' counters.
// -------------------------------------------------------------------------------------------------------
constexpr int kRingStages = 2;

__global__ void __launch_bounds__(kRowsTile) k_filter_rows_ring(const __grid_constant__ Plan P, uint64_t *__restrict__ keys,
                                                                int64_t key_cap, int32_t *__restrict__ counts)
{
    extern __shared__ __align__(128) float ring[];          // kRingStages tiles of 128 * (row_w_in | 1) floats
    __shared__ __align__(8) uint64_t full_bar[kRingStages];
    const int tid = static_cast<int>(threadIdx.x);
    const int rw = P.row_w_in;
    const int stage_floats = kRowsTile * (rw | 1);
    const long long total = static_cast<long long>(P.batch) * P.units_per_img;
    const long long G = gridDim.x;

    struct Unit {
        const LevelDesc *lv;
        const float *src;
        int img, r0, nrows;
        bool bulk;   // whole tile is a multiple of 16 bytes: one bulk copy; else plain loads at consumption time
    };
    auto unit_of = [&](long long w) {
        Unit u;
        u.img = static_cast<int>(w % P.batch);
        const int t = static_cast<int>(w / P.batch);
        int l = 0;
#pragma unroll
        for (int i = 1; i < YSB_MAX_LEVELS; ++i)
            if (i < P.L && t >= P.lv[i].unit_off) l = i;
        u.lv = &P.lv[l];
        const int rows_l = (l + 1 < P.L ? P.lv[l + 1].cand_off : P.N) - u.lv->cand_off;
        u.r0 = (t - u.lv->unit_off) * kRowsTile;
        u.nrows = min(kRowsTile, rows_l - u.r0);
        u.src = u.lv->p0 + (static_cast<size_t>(u.img) * u.lv->img_rows + u.r0) * rw;
        u.bulk = ((u.nrows * rw) & 3) == 0 && (reinterpret_cast<uintptr_t>(u.src) & 15u) == 0;
        return u;
    };
    auto arm = [&](long long w, int s) {   // thread 0: one arrival (+ the tile's bytes) completes the stage's phase
        const Unit u = unit_of(w);
        const uint32_t bar = smem_u32(&full_bar[s]);
        if (u.bulk) {
            const uint32_t bytes = static_cast<uint32_t>(u.nrows * rw) * 4u;
            mbar_expect_tx(bar, bytes);
            bulk_g2s(smem_u32(ring + static_cast<size_t>(s) * stage_floats), u.src, bytes, bar);
        } else {
            mbar_arrive(bar);
        }
    };

    if (tid == 0) {
#pragma unroll
        for (int s = 0; s < kRingStages; ++s) mbar_init(smem_u32(&full_bar[s]), 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (tid == 0) {
#pragma unroll
        for (int s = 0; s < kRingStages; ++s) {
            const long long w = blockIdx.x + s * G;
            if (w < total) arm(w, s);
        }
    }
    int k = 0;
    for (long long w = blockIdx.x; w < total; w += G, ++k) {
        const int s = k % kRingStages;
        const uint32_t phase = static_cast<uint32_t>(k / kRingStages) & 1u;
        const Unit u = unit_of(w);
        float *tile = ring + static_cast<size_t>(s) * stage_floats;
        mbar_wait(smem_u32(&full_bar[s]), phase);
        int sstride = rw;
        if (!u.bulk) {   // odd shapes (CTA-uniform): scalar loads into a tile padded to an odd stride
            sstride = rw | 1;
            const int nfl = u.nrows * rw;
            for (int e = tid; e < nfl; e += kRowsTile) {
                const int row = e / rw, col = e - row * rw;
                tile[row * sstride + col] = ldg_stream1(u.src + e);
            }
            __syncthreads();
        }
        rows_scan_emit(P, *u.lv, u.img, tile, sstride, u.nrows, u.r0, tid, keys, key_cap, counts);
        __syncthreads();   // every thread is done reading the stage
        if (tid == 0) {
            const long long wn = w + kRingStages * G;
            // (generic-proxy stores of an odd-shaped tile are ordered before the engine's next write into the stage)
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            if (wn < total) arm(wn, s);
        }
    }
}

#endif  // YSB_PROFILING_VARIANTS

// -------------------------------------------------------------------------------------------------------
// mutil_label: true -- one record per (candidate, class) whose score reaches the class threshold
// (trainer/eval_yolov5.py:276-279, eval_yolov7.py:230-233, eval_yolox.py:217-220, eval_yolov8.py:184-187,
// eval_fcos.py:246-250).  False in every shipped yaml, so this kernel favours simplicity: one thread per candidate,
// every class evaluated literally (sigmoid, multiply) twice -- once to count, once to write -- any input layout.
// -------------------------------------------------------------------------------------------------------
template <typename T, bool NHWC, bool WIDE = false>
__global__ void __launch_bounds__(256) k_filter_multilabel(const __grid_constant__ Plan P, uint64_t *__restrict__ keys,
                                                           int64_t key_cap, int32_t *__restrict__ counts)
{
    const int img = blockIdx.x;
    const int cand = blockIdx.y * blockDim.x + threadIdx.x;
    const bool active = cand < P.N;
    const bool decoded = P.input_kind == YSB_INPUT_DECODED_ROWS;
    const T *cls = nullptr;
    size_t cstride = 1;
    float mult = 1.0f;
    if (active) {
        const int l = find_level(P, cand);
        const LevelDesc &lv = P.lv[l];
        const int r = cand - lv.cand_off;
        float objv = 0.0f;
        if (NHWC || P.layout == LAYOUT_PLANES) {   // planes-family raw heads, NCHW or NHWC
            const int a = r / lv.hw, pos = r - a * lv.hw;
            cls = head_elem<T, NHWC>(lv, lv.p0, P.A, P.cls_nch, img, a, pos, P.cls_ch);
            cstride = static_cast<size_t>(head_step<NHWC>(lv));
            if (P.use_obj) objv = ldg_head(head_elem<T, NHWC>(lv, P.obj_src == 2 ? lv.p2 : lv.p0, P.A, P.obj_nch, img, a, pos, P.obj_ch));
        } else {
            const T *row = head_ptr<T>(lv.p0) + (static_cast<size_t>(img) * lv.img_rows + r) * P.row_w_in;
            cls = row + P.cls_col_in;
            if (P.use_obj)
                objv = P.obj_src == 1 ? ldg_head(head_ptr<T>(P.lv[0].p1) + (static_cast<size_t>(img) * P.N + cand) * P.reg_row_w + 4)
                                      : ldg_head(row + P.obj_col_in);
        }
        if (P.use_obj) mult = decoded ? objv : sigmoid_ref(objv);
    }
    auto score_of = [&](int k, float &sk) {
        const float c = ldg_head(cls + static_cast<size_t>(k) * cstride);
        sk = decoded ? c : sigmoid_ref(c);
        return P.use_obj ? __fmul_rn(sk, mult) : sk;
    };
    auto passes = [&](float p) { return P.multi_strict ? (p > P.cls_thr) : (p >= P.cls_thr); };
    int n = 0, npre = 0;
    uint32_t smax_bits = 0u, smin_inv = 0u;
    if (active) {
        float smax = -INFINITY, pmax = -INFINITY;
        for (int k = 0; k < P.C; ++k) {
            float sk;
            const float p = score_of(k, sk);
            smax = fmaxf(smax, sk);
            pmax = fmaxf(pmax, p);
            if (sk > P.pre_thr) ++npre;
            if (passes(p)) {
                ++n;
                const uint32_t sb = __float_as_uint(p);
                smax_bits = max(smax_bits, sb);
                smin_inv = max(smin_inv, ~sb);
            }
        }
        bool pre = true;
        switch (P.pre_kind) {
        case PRE_OBJ: pre = mult >= P.conf_thr; break;
        case PRE_OBJ_X_MAX: pre = pmax >= P.conf_thr; break;
        case PRE_MAXCLS: pre = smax >= P.cls_thr; break;
        case PRE_ANY_GT: pre = smax > P.pre_thr; break;
        default: break;
        }
        if (!pre) { n = 0; smax_bits = 0u; smin_inv = 0u; }
        if (P.pre_kind != PRE_ANY_GT) npre = 0;
    }
    // warp-aggregated reservation of n slots per thread
    const unsigned lane = threadIdx.x & 31u;
    int incl = n;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const int v = __shfl_up_sync(0xffffffffu, incl, d);
        if (lane >= static_cast<unsigned>(d)) incl += v;
    }
    const int total = __shfl_sync(0xffffffffu, incl, 31);
    int32_t *cnt = counts + img * 4;
    const int tp = __reduce_add_sync(0xffffffffu, npre);
    if (lane == 0 && tp) atomicAdd(cnt + 1, tp);  // FCOS: pairs above pre_nms_thresh (eval_fcos.py:246)
    if (total == 0) return;
    const uint32_t wmax = __reduce_max_sync(0xffffffffu, smax_bits);
    const uint32_t wmin = __reduce_max_sync(0xffffffffu, smin_inv);
    int base = 0;
    if (lane == 0) {
        base = atomicAdd(cnt, total);
        atomicMax(reinterpret_cast<unsigned int *>(cnt + 2), wmax);
        atomicMax(reinterpret_cast<unsigned int *>(cnt + 3), wmin);
    }
    base = __shfl_sync(0xffffffffu, base, 0);
    if (n > 0) {
        int64_t at = static_cast<int64_t>(base) + (incl - n);
        uint64_t *dst = keys + static_cast<int64_t>(img) * key_cap;
        for (int k = 0; k < P.C; ++k) {
            float sk;
            const float p = score_of(k, sk);
            if (passes(p)) {
                if (at < key_cap) dst[at] = pack_key<WIDE>(p, static_cast<uint32_t>(P.cand_base + cand), static_cast<uint32_t>(k));
                ++at;
            }
        }
    }
}

// -------------------------------------------------------------------------------------------------------
// host launcher
// -------------------------------------------------------------------------------------------------------
#ifdef YSB_PROFILING_VARIANTS
#include "filter_variants_launch.inc"
#endif

// planes layout (NCHW heads).  WIDE: the sort-key layout of plans with more than 1024 classes
template <typename T, bool WIDE>
static cudaError_t launch_planes(const Plan &P, int vec, uint64_t *d_keys, int64_t key_cap, int32_t *d_counts,
                                 cudaStream_t stream)
{
    cudaError_t e = cudaSuccess;
    // image-fastest grids: CTAs that run at the same time append to different images' counters
    if (vec == 4) {
        // every level 128-bit loadable (the common case): 9 loads of 128 bits in flight per thread (YOLOv5 / YOLOX:
        // 80 classes + objectness = 9 batches of 9), 76 registers, 6 CTAs of 128 threads per SM
        const dim3 gv4(P.batch, (P.units_per_img + 127) / 128);
#ifdef YSB_PROFILING_VARIANTS
        if (sizeof(T) == 4) {   // profiling build: YSB_K1_CARVEOUT=<percent of the SM's shared memory> as the kernel's preferred carve-out
            static int pct = -2;
            if (pct == -2) { const char *ev = getenv("YSB_K1_CARVEOUT"); pct = ev ? atoi(ev) : -1; }
            if (pct >= 0) {
                e = cudaFuncSetAttribute(k_filter_planes_v4<T, 9, 128, 6, 0, WIDE>, cudaFuncAttributePreferredSharedMemoryCarveout, pct);
                if (e != cudaSuccess) return e;
            }
        }
#endif
        k_filter_planes_v4<T, 9, 128, 6, 0, WIDE><<<gv4, 128, 0, stream>>>(P, d_keys, key_cap, d_counts);
    } else if (vec == 1) {
        const dim3 grid(P.batch, (P.units_per_img + 255) / 256);
        k_filter_planes<T, 1, 8, 256, 1, 0, 0, WIDE><<<grid, 256, 0, stream>>>(P, d_keys, key_cap, d_counts);
    } else {
        // levels that are not all 128-bit loadable (FCOS' 5x5 map): generic kernel, 128-thread CTAs, 12 loads of
        // 128 bits in flight per thread (96 registers, 5 CTAs/SM), 256-byte L2 prefetch
        const dim3 grid128(P.batch, (P.units_per_img + 127) / 128);
        k_filter_planes<T, 4, 12, 128, 5, 1, 0, WIDE><<<grid128, 128, 0, stream>>>(P, d_keys, key_cap, d_counts);
    }
    return e;
}

template <typename T>
static cudaError_t launch_filter_t(const Plan &P, int vec, uint64_t *d_keys, int64_t key_cap, int32_t *d_counts,
                                   cudaStream_t stream)
{
    cudaError_t e = cudaSuccess;
    const bool wide = wide_keys(P.C);
    if (P.multi_label) {
        const dim3 grid(P.batch, (P.N + 255) / 256);
        if (P.layout == LAYOUT_ROWS_NHWC) k_filter_multilabel<T, true><<<grid, 256, 0, stream>>>(P, d_keys, key_cap, d_counts);
        else if (wide) k_filter_multilabel<T, false, true><<<grid, 256, 0, stream>>>(P, d_keys, key_cap, d_counts);
        else k_filter_multilabel<T, false><<<grid, 256, 0, stream>>>(P, d_keys, key_cap, d_counts);
        return cudaGetLastError();
    }
    if (P.layout != LAYOUT_PLANES && !rows_fit_tile(P.row_w_in)) {
        // rows wider than the shared tile (never channels-last: the ABI refuses those)
        const dim3 grid(P.batch, P.units_per_img);
        if (wide) k_filter_rows_wide<T, true><<<grid, kRowsTile, 0, stream>>>(P, d_keys, key_cap, d_counts);
        else k_filter_rows_wide<T, false><<<grid, kRowsTile, 0, stream>>>(P, d_keys, key_cap, d_counts);
        return cudaGetLastError();
    }
    if (P.layout == LAYOUT_PLANES && wide) {   // (the profiling variants pack narrow keys)
        e = launch_planes<T, true>(P, vec, d_keys, key_cap, d_counts, stream);
        return e != cudaSuccess ? e : cudaGetLastError();
    }
#ifdef YSB_PROFILING_VARIANTS
    if (sizeof(T) == 4 && P.layout != LAYOUT_ROWS_NHWC) {   // the variants read float32 NCHW heads; 16-bit and NHWC heads run the product kernels
        bool handled = false;
        e = launch_filter_variant(P, vec, d_keys, key_cap, d_counts, stream, &handled);
        if (handled) return e;
    }
#endif
    if (P.layout == LAYOUT_PLANES) {
        e = launch_planes<T, false>(P, vec, d_keys, key_cap, d_counts, stream);
        if (e != cudaSuccess) return e;
    } else {
        const size_t smem = static_cast<size_t>(kRowsTile) * (P.row_w_in | 1) * sizeof(T);
#ifdef YSB_PROFILING_VARIANTS
        // persistent ring kernel when two CTAs with kRingStages tiles each fit an SM and the tensors allow bulk copies
        // (16-byte aligned bases, image strides that keep every image's first row 16-byte aligned)
        static int ring_env = -1;
        if (ring_env < 0) { const char *ev = getenv("YSB_ROWS_RING"); ring_env = ev ? atoi(ev) : 0; }
        bool ring_ok = sizeof(T) == 4 && P.layout != LAYOUT_ROWS_NHWC && ring_env != 0 && kRingStages * smem <= 110u * 1024u;
        for (int l = 0; l < P.L && ring_ok; ++l)
            ring_ok = (reinterpret_cast<uintptr_t>(P.lv[l].p0) & 15u) == 0 &&
                      ((static_cast<long long>(P.lv[l].img_rows) * P.row_w_in) & 3) == 0;
        if (ring_ok) {
            const size_t rsmem = kRingStages * smem;
            e = cudaFuncSetAttribute(k_filter_rows_ring, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(rsmem));
            if (e != cudaSuccess) return e;
            int dev = 0, sms = 148;
            if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
            const long long total = static_cast<long long>(P.batch) * P.units_per_img;
            const long long slots = static_cast<long long>(sms) * (rsmem <= 74u * 1024u ? 3 : 2);
            k_filter_rows_ring<<<static_cast<unsigned>(total < slots ? total : slots), kRowsTile, rsmem, stream>>>(P, d_keys, key_cap, d_counts);
            return cudaGetLastError();
        }
#endif
        const dim3 grid(P.batch, P.units_per_img);
        // Staging (bit 0): one bulk copy per tile for rows with an even float stride (RetinaNet, 84-float decoded rows),
        // cp.async for odd strides (YOLOv7's 85-float rows).  Measured in the 4-lane pipeline on B200: RetinaNet b=64
        // 207.5 k -> 214 k images/s with the bulk copy (three A/B pairs), YOLOv7 b=64 634 k -> 610 k.  Bit 1 (128-bit
        // shared loads + four scan chains) measured neutral (208.7 k / 213.1 k) and is only reachable in profiling builds.
        // Two threads per row (256-thread CTAs, halves merged by shuffle) measured 1.7x SLOWER (RetinaNet 216 k -> 124 k,
        // YOLOv7 642 k -> 366 k) and was removed.
        int flags = (P.row_w_in & 1) ? 0 : 1;
#ifdef YSB_PROFILING_VARIANTS
        {
            static int fenv = -2;
            if (fenv == -2) { const char *ev = getenv("YSB_ROWS_FLAGS"); fenv = ev ? atoi(ev) : -1; }
            if (fenv >= 0 && sizeof(T) == 4) flags = fenv;
        }
#endif
        // NHWC planes-family heads: the same kernel over each level's (H*W*A, K) row matrix, rows mapped to candidates
        auto kern = P.layout == LAYOUT_ROWS_NHWC ? k_filter_rows<T, true> : k_filter_rows<T, false>;
        if (smem > 48 * 1024) {
            e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
            if (e != cudaSuccess) return e;
        }
        kern<<<grid, kRowsTile, smem, stream>>>(P, d_keys, key_cap, d_counts, flags);
    }
    return cudaGetLastError();
}

// zero_counts = false: append to the key lists / counters a previous pass left (test-time-augmentation passes)
cudaError_t launch_filter(const Plan &P, int vec, uint64_t *d_keys, int64_t key_cap, int32_t *d_counts,
                          cudaStream_t stream, bool zero_counts, int dtype)
{
    cudaError_t e = cudaSuccess;
    if (zero_counts) e = cudaMemsetAsync(d_counts, 0, sizeof(int32_t) * 4 * static_cast<size_t>(P.batch), stream);
    if (e != cudaSuccess) return e;
    if (P.batch == 0 || P.N == 0) return cudaSuccess;
    switch (dtype) {
    case YSB_F16: return launch_filter_t<__half>(P, vec, d_keys, key_cap, d_counts, stream);
    case YSB_BF16: return launch_filter_t<__nv_bfloat16>(P, vec, d_keys, key_cap, d_counts, stream);
    default: return launch_filter_t<float>(P, vec, d_keys, key_cap, d_counts, stream);
    }
}

}  // namespace ysb
