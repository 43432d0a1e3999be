// nms_kernel.cu -- K2: per-image top-k selection + sort + greedy class-aware NMS + box post-filter.
//
// Replaces, per image, trainer/eval_yolov5.py:293-316 (class offset, utils.nms.numba_nms, max_det truncation,
// postprocess_bbox count filter, row gather) and the same tail in the other evaluators; the NMS itself is
// utils/nms.py:10-27 with the IoU of utils/bbox_tools.py:12-35.
//
// The reference runs the greedy loop over all M survivors (O(K*M), ~14 s per image at M = 25 k) and truncates to
// max_det afterwards.  Greedy NMS is prefix-stable, so this kernel visits candidates in the reference's order
// (score desc, candidate asc) and stops at max_det keeps:
//   1. pick a score threshold for the next tranche of best keys -- the FIRST tranche is sized for a sort with one element
//      per thread (most images reach max_det inside it), later ones are larger: radix descent over shared-memory
//      histograms of the normalised 64-bit keys -- of a strided SAMPLE of them when the image has many survivors (the exact
//      gather that follows counts what the threshold really selects and falls back to the exact descent if it overflows),
//   2. gather those keys (one pass over the image's key list, one shared-memory reservation per warp and 8 ballots),
//      bitonic-sort them (registers + shuffles, shared memory only for strides >= 32), decode their boxes (4 channels
//      each) from the head tensors as far as the walk gets,
//   3. walk them 128 at a time: every candidate against the kept list, in-chunk predecessor masks, greedy resolution by
//      one warp, append.  While all boxes seen are finite and span <= 4095 px in x, classes cannot interact through the
//      reference's cls * 4096 offset, and a candidate is only tested against the kept / chunk boxes of its own class
//      bucket (bit masks per bucket); otherwise against all of them (4-8 threads per candidate),
//   4. if fewer than max_det boxes are kept and candidates remain, select the next tranche and continue,
//   5. postprocess_bbox count filter / RetinaNet merge (streamed over ALL survivors in blocks, bucketed by class) /
//      remove_small_boxes, ordered write of the rows -- to the caller's buffer or, in a multi-GPU detection gather, into
//      every peer's receive slot over NVLink.
// One CTA per image.  Two flavours of the CTA (launch_any): 1024 threads (lowest latency: small batches, YOLOv8's DFL
// decode, very long key lists) and 512 threads (from 32 images up: half of the SM's registers stay free for the filter
// CTAs of the next batches, and two CTAs fit an SM when there are more images than SMs).  The shared-memory footprint
// (94 KB at max_det <= 320) is kept under the 100 KB carve-out step on purpose, see NmsSmem.
// The heads are read only by the box decode (decode_boxes): the kernel is templated on their element type T, and the
// float instantiations are those of the float32-only engine.
#include <cstdlib>

#include "ysb_internal.cuh"

namespace ysb {

constexpr int kTranche = 2048;      // keys selected, sorted and walked at a time
constexpr int kMinTranche = 512;    // a tranche smaller than this is only taken when nothing else is left
constexpr int kSampleTarget = 1024; // size a later tranche is aimed at when its threshold comes from a sample
template <int THREADS> constexpr int kFirstTarget = THREADS >= 1024 ? 640 : (THREADS * 13) / 16;  // first tranche
constexpr int kDigitBits = 11;
constexpr int kBins = 1 << kDigitBits;
constexpr int kChunk = 128;         // candidates resolved per step of the greedy walk
constexpr int kChunkWords = kChunk / 32;
// class buckets (cls & (buckets - 1)) of the kept-slot / chunk-slot bit masks of the walk; sized so that the masks fit the
// shared arrays they alias (NmsSmem)
template <int KEEP> constexpr int kMaskBuckets = KEEP <= 320 ? 128 : 32;
constexpr int kKeyBatch = 8;        // independent 64-bit key loads in flight per thread in the selection passes

// Phase timestamps of image 0..63 (profiling builds only: -DYSB_K2_TIMING), read back by ysb_debug_k2_timing().
#ifdef YSB_K2_TIMING
__device__ long long g_k2_timing[64][16];
#define K2_STAMP(slot) do { if (threadIdx.x == 0 && blockIdx.x < 64) g_k2_timing[blockIdx.x][slot] = clock64(); } while (0)
#define K2_ACC_BEGIN() k2_t0 = clock64()
#define K2_ACC(slot) do { const long long k2_t1 = clock64(); k2_acc[slot - 8] += k2_t1 - k2_t0; k2_t0 = k2_t1; } while (0)
#define K2_ACC_RESET() long long k2_acc[5] = {0, 0, 0, 0, 0}; long long k2_t0 = 0
#define K2_ACC_FLUSH() do { if (threadIdx.x == 0 && blockIdx.x < 64) for (int q = 0; q < 5; ++q) g_k2_timing[blockIdx.x][8 + q] = k2_acc[q]; } while (0)
#else
#define K2_ACC_BEGIN() do { } while (0)
#define K2_ACC(slot) do { } while (0)
#define K2_ACC_RESET() do { } while (0)
#define K2_ACC_FLUSH() do { } while (0)
#define K2_STAMP(slot) do { } while (0)
#endif

template <int KEEP>
struct NmsSmem {
    uint64_t keys[kTranche];
    float4 raw[kTranche];          // raw boxes of the tranche entries; post-filter: offset boxes of a survivor block
    // The walk's class-bucket masks live in arrays only the post-filter uses: the footprint must stay below the 100 KB
    // shared-memory carve-out step.  With the masks as separate fields (101 KB -> 132 KB carve-out, 32 KB less L1 for the
    // in-flight loads of the filter CTAs that share the SM) the 4-lane pipeline lost 11 % (YOLOv5s b=64 745 k -> 660 k
    // images/s, YOLOX b=256 1.93 M -> 1.75 M; aliased: 755 k / 2.02 M, A/B on one box).
    union {
        float area[kTranche];                                          // post-filter: areas of the offset boxes
        uint32_t kept_mask[kMaskBuckets<KEEP>][(KEEP + 31) / 32];      // walk: kept slots holding a box of the bucket
    };
    uint32_t hist[kBins];          // selection histograms; post-filter: class bucket bounds and cursors
    union {
        uint16_t order[kTranche];                                      // post-filter: survivor indices sorted by class
        uint32_t chunk_mask[kMaskBuckets<KEEP>][kChunkWords];          // walk: chunk slots holding a candidate of the bucket
    };
    float2 kept_x[KEEP];
    float2 kept_y[KEEP];
    float kept_a[KEEP];
    uint64_t kept_key[KEEP];
    float4 kept_raw[KEEP];
    float kept_acc[KEEP][5];       // RetinaNet merge: score-weighted box sums and the weight sum
    uint16_t kept_cnt[KEEP];       // post-filter: survivors overlapping the kept box by more than the threshold
    uint8_t kept_flag[KEEP];
    float2 chunk_x[kChunk];
    float2 chunk_y[kChunk];
    float chunk_a[kChunk];
    uint32_t chunk_pred[kChunk][kChunkWords];  // row j: earlier candidates i < j of the chunk that suppress j
    uint32_t keep_words[kChunkWords];
    uint8_t chunk_alive[kChunk];
    int run_lo, run_hi, run_bad;   // x-span (order-preserving ints) of every box decoded so far; a non-finite one was seen
    uint32_t warp_tmp[32];
    int n_sel;
    int sel_digit;
    int sel_above;
    int span_lo, span_hi;
};

// Arguments of the array flavour (utils.numba_nms / utils.gpu_nms on one explicit box array).
struct ArrayArgs {
    const float4 *boxes;   // (m) xyxy
    BoxSoA kept;           // global workspace (m boxes): the keep list is unbounded here
    int32_t *keep;         // out: kept indices, visiting order
    int32_t *keep_cnt;     // out
    int iou_kind, cmp;
    float thr32;           // torch compares float32 IoUs against the threshold rounded to float32
};

// One pair test against entry i of a SoA box list (generic: any IoU flavour of the array kernels).
template <bool ARRAY>
__device__ __forceinline__ bool pair_hit(const BoxSoA &list, int i, const OffBox &b, const IouThr &t, const ArrayArgs &aa)
{
    if (!ARRAY) return iou_reaches_staged<false>(list, i, b, t);
    if (aa.iou_kind == YSB_IOU_NUMBA_F64MIX)
        return aa.cmp == YSB_CMP_GT ? iou_reaches_staged<true>(list, i, b, t) : iou_reaches_staged<false>(list, i, b, t);
    const OffBox a = soa_load(list, i);
    const float v = iou_kind_f32(aa.iou_kind, make_float4(a.x1, a.y1, a.x2, a.y2), make_float4(b.x1, b.y1, b.x2, b.y2));
    return aa.cmp == YSB_CMP_GT ? (v > aa.thr32) : (v >= aa.thr32);
}

// The pair test after the x interval of entry i has been loaded and found to overlap b's (numba flavour only).
template <bool ARRAY>
__device__ __forceinline__ bool pair_hit_after_x(const BoxSoA &list, int i, float dw, const OffBox &b, const IouThr &t,
                                                 const ArrayArgs &aa)
{
    const float2 ay = list.y[i];
    const float dh = __fsub_rn(fminf(ay.y, b.y2), fmaxf(ay.x, b.y1));
    if (!(dh > 0.0f)) return false;
    const bool strict = ARRAY && aa.cmp == YSB_CMP_GT;
    return strict ? iou_decide<true>(dw, dh, list.area[i], b.area, t) : iou_decide<false>(dw, dh, list.area[i], b.area, t);
}

// Does box b hit any of the entries first, first + step, ... < end of the list?  Four independent x-interval loads are
// in flight per thread; with the 4096-px class offset nearly every pair is rejected by that single 64-bit load.
template <bool ARRAY>
__device__ __forceinline__ bool any_hit_strided(const BoxSoA &list, int first, int step, int end, const OffBox &b,
                                                const IouThr &t, const ArrayArgs &aa)
{
    const bool fast = t.positive && (!ARRAY || aa.iou_kind == YSB_IOU_NUMBA_F64MIX);
    bool hit = false;
    if (fast) {
        for (int k0 = first; k0 < end; k0 += 4 * step) {
            float dw[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const int k = k0 + q * step;
                const float2 ax = k < end ? list.x[k] : make_float2(0.0f, -1.0f);
                dw[q] = k < end ? __fsub_rn(fminf(ax.y, b.x2), fmaxf(ax.x, b.x1)) : -1.0f;
            }
            // the rare x-overlaps go through ONE copy of the slow path (float64 IoU decision): keeps the loop body small
            unsigned m = (dw[0] > 0.0f ? 1u : 0u) | (dw[1] > 0.0f ? 2u : 0u) | (dw[2] > 0.0f ? 4u : 0u) | (dw[3] > 0.0f ? 8u : 0u);
            while (m) {
                const int q = __ffs(m) - 1;
                m &= m - 1u;
                const float d = q == 0 ? dw[0] : (q == 1 ? dw[1] : (q == 2 ? dw[2] : dw[3]));
                hit |= pair_hit_after_x<ARRAY>(list, k0 + q * step, d, b, t, aa);
            }
        }
    } else {
        for (int k = first; k < end; k += step) hit |= pair_hit<ARRAY>(list, k, b, t, aa);
    }
    return hit;
}

__device__ __forceinline__ uint64_t norm_key(uint64_t key, uint32_t smin)
{
    return (static_cast<uint64_t>(static_cast<uint32_t>(key >> 32) - smin) << 32) | (key & 0xffffffffull);
}

// Block-wide radix descent over the normalised keys nk <= hi_incl, visiting every `stride`-th key of the list: returns
// a lower bound `lo` such that {lo <= nk <= hi_incl} holds -- by the (sampled) counts -- at least `want` keys, or
// everything that is left, and at most `cap`.  The smallest such set at the coarsest digit that resolves it is taken.
// stride == 1: exact counts.  stride > 1: an estimate; the caller's exact gather pass validates it.
template <int THREADS, int KEEP>
__device__ uint64_t select_lower_bound(NmsSmem<KEEP> &S, const uint64_t *__restrict__ keys, int M, uint32_t smin,
                                       uint64_t hi_incl, int nbits, int stride, int want, int cap)
{
    const int tid = threadIdx.x;
    int sh = nbits > kDigitBits ? nbits - kDigitBits : 0;  // shift of the current digit
    int width = nbits - sh;                                // bits in the current digit
    uint64_t prefix = 0;                                   // value of nk >> (sh + width) along the descent path
    bool have_prefix = false;
    int acc = 0;                                           // (sampled) keys already covered above the path
    const int ms = (M + stride - 1) / stride;              // sample size
    for (;;) {
        for (int i = tid; i < kBins; i += THREADS) S.hist[i] = 0;
        if (tid == 0) { S.sel_digit = -1; S.n_sel = 0; S.sel_above = 0; }
        __syncthreads();
        const int top = sh + width;
        const uint32_t dmask = (1u << width) - 1u;
        for (int i0 = 0; i0 < ms; i0 += kKeyBatch * THREADS) {
            uint64_t kk[kKeyBatch];
#pragma unroll
            for (int q = 0; q < kKeyBatch; ++q) {
                const int i = i0 + q * THREADS + tid;
                kk[q] = i < ms ? __ldg(keys + static_cast<int64_t>(i) * stride) : 0ull;
            }
#pragma unroll
            for (int q = 0; q < kKeyBatch; ++q) {
                if (i0 + q * THREADS + tid >= ms) continue;
                const uint64_t nk = norm_key(kk[q], smin);
                if (nk <= hi_incl && (!have_prefix || (nk >> top) == prefix))
                    atomicAdd(&S.hist[static_cast<uint32_t>(nk >> sh) & dmask], 1u);
            }
        }
        __syncthreads();
        // suffix sums S(d) = #keys with digit >= d; thread t owns digits PER*t .. PER*t + PER - 1
        constexpr int PER = kBins / THREADS;
        uint32_t h[PER];
        uint32_t part = 0;
#pragma unroll
        for (int q = 0; q < PER; ++q) { h[q] = S.hist[PER * tid + q]; part += h[q]; }
        uint32_t incl = part;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const uint32_t v = __shfl_down_sync(0xffffffffu, incl, d);
            if ((tid & 31) + d < 32) incl += v;
        }
        if ((tid & 31) == 0) S.warp_tmp[tid >> 5] = incl;
        __syncthreads();
        uint32_t above = 0;
        for (int w = (tid >> 5) + 1; w < THREADS / 32; ++w) above += S.warp_tmp[w];
        uint32_t s_hi = incl - part + above;  // S(PER*t + PER)
        const uint32_t need = static_cast<uint32_t>(want > acc ? want - acc : 0);
        // d_a = largest digit with S(d_a) >= need
#pragma unroll
        for (int q = PER - 1; q >= 0; --q) {
            const uint32_t s_lo = s_hi + h[q];  // S(PER*t + q)
            if (s_lo >= need && s_hi < need) { S.sel_digit = PER * tid + q; S.n_sel = static_cast<int>(s_lo); S.sel_above = static_cast<int>(s_hi); }
            s_hi = s_lo;
        }
        __syncthreads();
        const int da = S.sel_digit, covered = acc + S.n_sel, abv = acc + S.sel_above;
        __syncthreads();
        const uint64_t base = have_prefix ? (prefix << top) : 0ull;
        if (da < 0) return base;  // fewer than `want` keys under this prefix: take them all
        if (covered <= cap || sh == 0) return base | (static_cast<uint64_t>(da) << sh);
        // digit d_a alone overflows the tranche: refine inside it
        prefix = (have_prefix ? (prefix << width) : 0ull) | static_cast<uint64_t>(da);
        have_prefix = true;
        acc = abv;
        const int nw = sh < kDigitBits ? sh : kDigitBits;
        sh -= nw;
        width = nw;
    }
}

// Block-wide gather of the keys with lo <= norm_key <= hi_incl into S.keys[at0 ...) (arrival order); returns at0 + their
// count (entries beyond kTranche are counted, not stored).  One pass over the image's key list.
template <int THREADS, int KEEP>
__device__ int gather_range(NmsSmem<KEEP> &S, const uint64_t *__restrict__ keys, int M, uint32_t smin, uint64_t lo,
                            uint64_t hi_incl, int at0)
{
    const int tid = threadIdx.x;
    if (tid == 0) S.n_sel = at0;
    __syncthreads();
    for (int i0 = 0; i0 < M; i0 += kKeyBatch * THREADS) {
        uint64_t kk[kKeyBatch];
#pragma unroll
        for (int q = 0; q < kKeyBatch; ++q) {
            const int i = i0 + q * THREADS + tid;
            kk[q] = i < M ? __ldg(keys + i) : 0ull;
        }
        // one shared-memory reservation per warp and batch (a reservation per ballot serialised ~M/32 atomics on one
        // address: with ~8 % of the keys selected nearly every ballot is non-empty)
        unsigned bal[kKeyBatch];
        int warp_total = 0;
#pragma unroll
        for (int q = 0; q < kKeyBatch; ++q) {
            const uint64_t nk = norm_key(kk[q], smin);
            const bool in = (i0 + q * THREADS + tid < M) && nk >= lo && nk <= hi_incl;
            bal[q] = __ballot_sync(0xffffffffu, in);
            warp_total += __popc(bal[q]);
        }
        if (warp_total) {
            int base = 0;
            if ((tid & 31) == 0) base = atomicAdd(&S.n_sel, warp_total);
            base = __shfl_sync(0xffffffffu, base, 0);
            const unsigned below = (1u << (tid & 31)) - 1u;
#pragma unroll
            for (int q = 0; q < kKeyBatch; ++q) {
                if ((bal[q] >> (tid & 31)) & 1u) {
                    const int at = base + __popc(bal[q] & below);
                    if (at < kTranche) S.keys[at] = kk[q];
                }
                base += __popc(bal[q]);
            }
        }
    }
    __syncthreads();
    const int n = S.n_sel;
    __syncthreads();
    return n;
}

// Descending sort of keys[0..n) (n <= THREADS*E) by a bitonic network held in registers: element i = tid + THREADS*r
// lives in register r of thread tid.  Strides >= THREADS are thread-local, strides < 32 use warp shuffles, only strides
// 32..THREADS/2 go through shared memory.  Slots beyond n sort as 0 (smaller than any real key).
template <int THREADS, int E, int DR>
__device__ __forceinline__ void local_stage(uint64_t (&v)[E], int tid, int k)
{
#pragma unroll
    for (int r = 0; r < E; ++r) {
        if ((r & DR) == 0 && r + DR < E) {
            const bool desc = ((tid + THREADS * r) & k) == 0;
            uint64_t &a = v[r], &b = v[(r + DR) % E];
            const uint64_t hi = a > b ? a : b, lo = a > b ? b : a;
            a = desc ? hi : lo;
            b = desc ? lo : hi;
        }
    }
}

template <int THREADS, int E>
__device__ void bitonic_sort_desc(uint64_t *keys, int n)
{
    const int tid = threadIdx.x;
    constexpr int n2 = THREADS * E;
    uint64_t v[E];
#pragma unroll
    for (int r = 0; r < E; ++r) {
        const int i = tid + THREADS * r;
        v[r] = i < n ? keys[i] : 0ull;
    }
    __syncthreads();
    for (int k = 2; k <= n2; k <<= 1) {
        for (int j = k >> 1; j > 0; j >>= 1) {
            if (j >= THREADS) {
                // thread-local stage: register pairs (r, r + j/THREADS); the pair distance is resolved at compile time so
                // that v[] stays in registers
                if (j == THREADS) local_stage<THREADS, E, 1>(v, tid, k);
                else if (j == 2 * THREADS) local_stage<THREADS, E, 2>(v, tid, k);
                else local_stage<THREADS, E, 4>(v, tid, k);
            } else if (j >= 32) {
#pragma unroll
                for (int r = 0; r < E; ++r) keys[tid + THREADS * r] = v[r];
                __syncthreads();
#pragma unroll
                for (int r = 0; r < E; ++r) {
                    const int i = tid + THREADS * r;
                    const uint64_t o = keys[i ^ j];
                    const bool take_max = ((i & j) == 0) == ((i & k) == 0);
                    v[r] = take_max ? (v[r] > o ? v[r] : o) : (v[r] > o ? o : v[r]);
                }
                __syncthreads();
            } else {
#pragma unroll
                for (int r = 0; r < E; ++r) {
                    const int i = tid + THREADS * r;
                    const uint64_t o = __shfl_xor_sync(0xffffffffu, v[r], j);
                    const bool take_max = ((i & j) == 0) == ((i & k) == 0);
                    v[r] = take_max ? (v[r] > o ? v[r] : o) : (v[r] > o ? o : v[r]);
                }
            }
        }
    }
#pragma unroll
    for (int r = 0; r < E; ++r) keys[tid + THREADS * r] = v[r];
    __syncthreads();
}

template <int THREADS>
__device__ __forceinline__ void sort_tranche(uint64_t *keys, int n)
{
    if (n <= THREADS) bitonic_sort_desc<THREADS, 1>(keys, n);
    else if (n <= 2 * THREADS) bitonic_sort_desc<THREADS, 2>(keys, n);
    else bitonic_sort_desc<THREADS, kTranche / THREADS>(keys, n);
}

// order-preserving float <-> int maps (signed integer compare == float compare; used for shared-memory atomicMin/Max)
__device__ __forceinline__ int float_ordered(float f)
{
    const int i = __float_as_int(f);
    return i ^ ((i >> 31) & 0x7fffffff);
}
__device__ __forceinline__ float ordered_float(int i) { return __int_as_float(i ^ ((i >> 31) & 0x7fffffff)); }

// Plan a merged candidate index belongs to (test-time-augmentation passes); cand becomes the index inside that pass.
__device__ __forceinline__ const Plan &pass_of(const Plan &P, const NoExtraPasses &, int &) { return P; }
__device__ __forceinline__ const Plan &pass_of(const Plan &P, const ExtraPasses &X, int &cand)
{
    int sel = -1;
#pragma unroll
    for (int i = 0; i < YSB_MAX_PASSES - 1; ++i)
        if (i < X.n && cand >= X.base[i]) sel = i;
    if (sel < 0) return P;
    cand -= X.base[sel];
    return X.p[sel];
}

// Raw boxes of the tranche entries [from, upto) into S.raw.  YOLOv8 raw heads: a box is 4 sides x 16 DFL bins = 64
// scattered loads; one thread per (candidate, side) keeps its 16 bin loads in flight together and runs the softmax
// expectation in registers (the decode kernel's bin order), the four sides of a candidate meet by shuffle -- THREADS/4
// boxes per DRAM round trip.  Every other layout: one thread per box.
template <bool ARRAY, typename EXTRA, int THREADS, int KEEP, typename T, bool NHWC, bool WIDE>
__device__ __forceinline__ void decode_boxes(NmsSmem<KEEP> &S, const Plan &P, const EXTRA &X, const ArrayArgs &aa, int img,
                                             int from, int upto, int &lo_x, int &hi_x, bool &bad)
{
    const int tid = threadIdx.x;
    auto span = [&](const float4 &b) {   // this thread's share of the x-span of the decoded boxes
        bad = bad || !(fabsf(b.x) <= 3.0e38f) || !(fabsf(b.z) <= 3.0e38f);
        lo_x = min(lo_x, float_ordered(b.x));
        hi_x = max(hi_x, float_ordered(b.z));
    };
    if (!ARRAY && P.family == YSB_YOLOV8 && P.input_kind == YSB_INPUT_RAW_HEADS) {
        for (int i0 = from; i0 < upto; i0 += THREADS / 4) {
            const int i = i0 + (tid >> 2), side = tid & 3;
            float sv = 0.0f;
            const bool ok = i < upto;
            if (ok) {
                int cand = static_cast<int>(key_cand<WIDE>(S.keys[i]));
                const Plan &Q = pass_of(P, X, cand);
                sv = v8_side_value<T, NHWC>(Q, img, cand, side);
            }
            const unsigned qb = (tid & 31) & ~3u;
            const float s0 = __shfl_sync(0xffffffffu, sv, qb), s1 = __shfl_sync(0xffffffffu, sv, qb + 1);
            const float s2 = __shfl_sync(0xffffffffu, sv, qb + 2), s3 = __shfl_sync(0xffffffffu, sv, qb + 3);
            if (ok && side == 0) {
                int c2 = static_cast<int>(key_cand<WIDE>(S.keys[i]));
                const Plan &Q = pass_of(P, X, c2);
                const float4 b = tta_undo(Q, v8_box_from_sides(Q, c2, s0, s1, s2, s3));
                S.raw[i] = b;
                span(b);
            }
        }
    } else {
        for (int i = from + tid; i < upto; i += THREADS) {
            int cand = static_cast<int>(key_cand<WIDE>(S.keys[i]));
            if (ARRAY) {
                S.raw[i] = __ldg(aa.boxes + cand);
            } else {
                const Plan &Q = pass_of(P, X, cand);
                const float4 b = candidate_xyxy<T, NHWC>(Q, img, cand);
                S.raw[i] = b;
                span(b);
            }
        }
    }
}

// EXTRA = NoExtraPasses (one set of heads) or ExtraPasses (TTA: boxes are decoded from the pass a candidate came from;
// thresholds / NMS settings are those of P, identical in every pass).
// WIDE: the sort-key layout of plans with more than 1024 classes (ysb_internal.cuh, KeyLayout)
template <bool ARRAY, typename EXTRA, int THREADS, int KEEP, typename T = float, bool NHWC = false, bool WIDE = false>
__global__ void __launch_bounds__(THREADS, 1024 / THREADS)
k_select_nms(const __grid_constant__ Plan P, const __grid_constant__ EXTRA X, const uint64_t *__restrict__ keys_all,
             int64_t key_cap, const int32_t *__restrict__ counts, float *__restrict__ dets,
             int32_t *__restrict__ det_idx, int32_t *__restrict__ det_cnt, const ArrayArgs aa,
             const __grid_constant__ GatherSink G)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    using Smem = NmsSmem<KEEP>;
    Smem &S = *reinterpret_cast<Smem *>(smem_raw);
    const int tid = threadIdx.x;
    const int img = blockIdx.x;
    const int32_t *cnt = counts + img * 4;
    const int64_t m64 = cnt[0];
    const int M = static_cast<int>(m64 < key_cap ? m64 : key_cap);
    if (M <= 0) {
        if (tid == 0) {
            if (ARRAY) *aa.keep_cnt = 0;
            else if (G.world == 0) det_cnt[img] = -1;  // no survivor: the reference appends None
        }
        if (!ARRAY && G.world > 0 && tid < G.world) {   // detection gather: the count goes to every rank's slot
            // peer `tid` must have consumed the previous use of this slot before its region is overwritten
            if (tid != G.rank && !spin_until_reached(G.my_ack + tid, *G.use)) atomicExch(G.err, 1u);
            G.cnt[tid][img] = -1;
            __threadfence_system();
            atomicAdd_system(G.arrived[tid], 1u);
        }
        return;
    }
    const BoxSoA kept_box = ARRAY ? aa.kept : BoxSoA{S.kept_x, S.kept_y, S.kept_a};
    const BoxSoA chunk_box{S.chunk_x, S.chunk_y, S.chunk_a};
    const uint64_t *keys = keys_all + static_cast<int64_t>(img) * key_cap;
    const uint32_t smax = static_cast<uint32_t>(cnt[2]);
    const uint32_t smin = ~static_cast<uint32_t>(cnt[3]);
    const int nbits = 32 + (smax > smin ? 32 - __clz(smax - smin) : 0);
    const int limit = P.topk_sqrt ? min(M, min(cnt[1], P.pre_nms_topk)) : M;
    const IouThr thr = make_iou_thr(P.iou_thr);
    const int max_det = P.max_det;
    // postprocess_bbox runs only for 1 < M < 3000 (FCOS: <= 300), trainer/eval_yolov5.py:306-307
    const bool window = !ARRAY && P.postprocess_bbox && M > 1 && M < P.window_hi;

    // class-bucket masks of the walk (phase A / B below); the selection passes that follow contain the barriers that
    // order this initialisation before the first use
    if (!ARRAY) {
        for (int i = tid; i < kMaskBuckets<KEEP> * ((KEEP + 31) / 32); i += THREADS) (&S.kept_mask[0][0])[i] = 0u;
        for (int i = tid; i < kMaskBuckets<KEEP> * kChunkWords; i += THREADS) (&S.chunk_mask[0][0])[i] = 0u;
        if (tid == 0) { S.run_lo = 0x7fffffff; S.run_hi = static_cast<int>(0x80000000u); S.run_bad = 0; }
    }
    int kept = 0, processed = 0, n_tranche = 0, decoded_upto = 0;
    bool whole = false;   // the (single) tranche in shared memory holds every survivor
    uint64_t last_lo = 0; // lower bound of the last tranche's normalised keys
    uint64_t hi_incl = ~0ull;
    for (;;) {
        K2_STAMP(0);
        K2_ACC_RESET();
        // ---- 1. threshold of the next tranche ---------------------------------------------------------------
        // Many survivors left: estimate it from every stride-th key (the list is in arrival order, i.e. unordered in
        // score), aiming above the minimum so that sampling noise rarely leaves the tranche short.
        uint64_t lo = 0;
        int n = 0;
        const int remaining = M - processed;
        // First tranche: aimed at what ONE sort element per thread holds (most images reach max_det inside it, and the
        // bitonic network over THREADS slots costs less than half of the next size); if the walk needs more, the later
        // tranches are large (fewer passes over the key list).
        const bool first = processed == 0;
        const int take_all = first ? THREADS : kTranche;       // this many keys or fewer: no selection pass
        const int target = first ? kFirstTarget<THREADS> : kSampleTarget;
        int stride = remaining > 4 * kTranche ? (remaining >= 32 * kTranche ? 32 : remaining / kTranche) : 1;
        for (;;) {
            if (remaining > take_all) {
                const int want = stride > 1 ? (target + stride - 1) / stride : (first ? target : kMinTranche);
                const int cap = stride > 1 ? (first ? THREADS : kTranche * 3 / 4) / stride : (first ? THREADS : kTranche);
                lo = select_lower_bound<THREADS, KEEP>(S, keys, M, smin, hi_incl, nbits, stride, want, cap);
            }
            K2_STAMP(1);
            // ---- gather {lo <= nk <= hi_incl}: one exact pass over the key list -----------------------------------
            n = gather_range<THREADS, KEEP>(S, keys, M, smin, lo, hi_incl, 0);
            if (n <= kTranche) break;
            stride = 1;  // the sampled threshold let too many keys through: redo with exact counts
        }
        K2_STAMP(2);
        n_tranche = n;
        whole = processed == 0 && n == M;
        last_lo = lo;
        // ---- 2. sort descending -----------------------------------------------------------------------------------
        sort_tranche<THREADS>(S.keys, n);
        const int n_use = min(n, limit - processed);
        K2_STAMP(3);
        decoded_upto = 0;  // boxes are decoded a batch at a time, only as far as the NMS walk gets
        // ---- 3. greedy NMS over the tranche, kChunk candidates at a time ------------------------------------------
        constexpr int TPC = THREADS / kChunk;  // threads per candidate
        for (int c0 = 0; c0 < n_use && kept < max_det; c0 += kChunk) {
            const int cn = min(kChunk, n_use - c0);
            K2_ACC_BEGIN();
            if (c0 + cn > decoded_upto) {
                // one batch = one DRAM round trip; a YOLOv8 box costs 64 loads + 4 softmax expectations, so only as many as
                // one round of (candidate, side) threads covers are decoded ahead of the walk
                const bool dfl = !ARRAY && P.family == YSB_YOLOV8 && P.input_kind == YSB_INPUT_RAW_HEADS;
                const int upto = min(n_use, decoded_upto + (dfl ? max(THREADS / 4, kChunk) : THREADS));
                int d_lo = 0x7fffffff, d_hi = static_cast<int>(0x80000000u);
                bool d_bad = false;
                decode_boxes<ARRAY, EXTRA, THREADS, KEEP, T, NHWC, WIDE>(S, P, X, aa, img, decoded_upto, upto, d_lo, d_hi, d_bad);
                decoded_upto = upto;
                if (!ARRAY) {
                    d_lo = __reduce_min_sync(0xffffffffu, d_lo);
                    d_hi = __reduce_max_sync(0xffffffffu, d_hi);
                    d_bad = __any_sync(0xffffffffu, d_bad);
                    if ((tid & 31) == 0) {
                        atomicMin(&S.run_lo, d_lo);
                        atomicMax(&S.run_hi, d_hi);
                        if (d_bad) S.run_bad = 1;
                    }
                }
                __syncthreads();
            }
            K2_ACC(8);
            // Class-aware walk: while every box seen so far is finite and the boxes span at most 4095 px in x, boxes of
            // different classes are disjoint once offset (see the post-filter below for the bound), i.e. a candidate can
            // only be suppressed by boxes of its own class -- found through per-class-bucket bit masks of the kept slots
            // and of the chunk slots instead of testing every pair.  Buckets are cls & 127 (& 31): classes sharing a bucket only
            // cost extra pair tests, the tests themselves are the exact ones.  Anything else: all pairs, as before.
            const bool cls_fast = !ARRAY && P.class_aware && thr.positive && !S.run_bad &&
                                  __fsub_rn(ordered_float(S.run_hi), ordered_float(S.run_lo)) <= 4095.0f;
            const int j = tid / TPC, sub = tid % TPC;
            const unsigned group = ((1u << TPC) - 1u) << ((tid & 31) / TPC * TPC);
            // phase A: TPC threads per candidate test it against the kept list
            {
                bool sup = false;
                OffBox ob{};
                const bool valid = j < cn;
                float score = 0.f;
                if (valid) {
                    const uint64_t key = S.keys[c0 + j];
                    score = key_score(key);
                    const float off = P.class_aware ? __fmul_rn(static_cast<float>(key_cls<WIDE>(key)), 4096.0f) : 0.0f;
                    ob = make_offbox(S.raw[c0 + j], off);
                    if (cls_fast) {
                        const uint32_t *km = S.kept_mask[key_cls<WIDE>(key) & (kMaskBuckets<KEEP> - 1)];
                        const int nw = (kept + 31) >> 5;
                        for (int wd = sub; wd < nw; wd += TPC) {
                            uint32_t m = km[wd];
                            while (m) {
                                const int i = 32 * wd + __ffs(m) - 1;
                                m &= m - 1u;
                                sup |= pair_hit<ARRAY>(kept_box, i, ob, thr, aa);
                            }
                        }
                        if (sub == 0) atomicOr(&S.chunk_mask[key_cls<WIDE>(key) & (kMaskBuckets<KEEP> - 1)][j >> 5], 1u << (j & 31));
                    } else {
                        sup = any_hit_strided<ARRAY>(kept_box, sub, TPC, kept, ob, thr, aa);
                    }
                }
                const unsigned bal = __ballot_sync(0xffffffffu, sup);
                if (sub == 0) {
                    // a zero score is never picked by "while sum > 0" (utils/nms.py:16): it is neither kept nor a suppressor
                    S.chunk_alive[j] = valid && !(bal & group) && score > 0.0f;
                    if (valid) soa_store(chunk_box, j, ob);
                }
            }
            __syncthreads();
            K2_ACC(9);
            // phase B: in-chunk predecessor masks, pred[j] bit i (i < j) = IoU(i, j) reaches the threshold, both alive
            bool conflict;
            {
                uint32_t w[kChunkWords];
#pragma unroll
                for (int c = 0; c < kChunkWords; ++c) w[c] = 0u;
                if (cls_fast) {
                    if (j < cn && S.chunk_alive[j]) {
                        const OffBox bj = soa_load(chunk_box, j);
                        const uint32_t *cm = S.chunk_mask[key_cls<WIDE>(S.keys[c0 + j]) & (kMaskBuckets<KEEP> - 1)];
                        for (int wd = sub; wd <= (j >> 5); wd += TPC) {
                            uint32_t m = cm[wd];
                            if (wd == (j >> 5)) m &= (1u << (j & 31)) - 1u;   // earlier candidates only
                            while (m) {
                                const int i = 32 * wd + __ffs(m) - 1;
                                m &= m - 1u;
                                if (!S.chunk_alive[i]) continue;
                                if (pair_hit<ARRAY>(chunk_box, i, bj, thr, aa)) {
#pragma unroll
                                    for (int c = 0; c < kChunkWords; ++c)   // (static register index: no local memory)
                                        w[c] |= (i >> 5) == c ? 1u << (i & 31) : 0u;
                                }
                            }
                        }
                    }
                } else if (j < cn && S.chunk_alive[j]) {
                    const OffBox bj = soa_load(chunk_box, j);
                    const bool fast = thr.positive && (!ARRAY || aa.iou_kind == YSB_IOU_NUMBA_F64MIX);
                    for (int i0 = sub; i0 < j; i0 += 4 * TPC) {
                        float dw[4];
#pragma unroll
                        for (int q = 0; q < 4; ++q) {
                            const int i = i0 + q * TPC;
                            const float2 ax = i < j ? chunk_box.x[i] : make_float2(0.0f, -1.0f);
                            dw[q] = i < j ? __fsub_rn(fminf(ax.y, bj.x2), fmaxf(ax.x, bj.x1)) : -1.0f;
                        }
                        unsigned m = 0u;
#pragma unroll
                        for (int q = 0; q < 4; ++q)
                            if (i0 + q * TPC < j && (!fast || dw[q] > 0.0f)) m |= 1u << q;
                        while (m) {   // rare: ONE copy of the slow path
                            const int q = __ffs(m) - 1;
                            m &= m - 1u;
                            const int i = i0 + q * TPC;
                            if (!S.chunk_alive[i]) continue;
                            const float d = q == 0 ? dw[0] : (q == 1 ? dw[1] : (q == 2 ? dw[2] : dw[3]));
                            const bool hit = fast ? pair_hit_after_x<ARRAY>(chunk_box, i, d, bj, thr, aa)
                                                  : pair_hit<ARRAY>(chunk_box, i, bj, thr, aa);
                            if (hit) {
#pragma unroll
                                for (int c = 0; c < kChunkWords; ++c)   // (static register index: no local memory)
                                    w[c] |= (i >> 5) == c ? 1u << (i & 31) : 0u;
                            }
                        }
                    }
                }
                // OR the TPC partial masks of a candidate (xor-shuffles stay inside the aligned group of TPC lanes); hits
                // are rare, so most warps skip it
                if (__any_sync(0xffffffffu, (w[0] | w[1] | w[2] | w[3]) != 0u)) {
#pragma unroll
                    for (int c = 0; c < kChunkWords; ++c)
#pragma unroll
                        for (int d = 1; d < TPC; d <<= 1) w[c] |= __shfl_xor_sync(0xffffffffu, w[c], d);
                }
                uint32_t any_w = 0u;
#pragma unroll
                for (int c = 0; c < kChunkWords; ++c) {
                    if (sub == 0) S.chunk_pred[j][c] = w[c];
                    any_w |= w[c];
                }
                // the barrier that ends the phase also tells everybody whether the chunk has any in-chunk suppression
                conflict = __syncthreads_or(any_w != 0u) != 0;
            }
            K2_ACC(10);
            // phase C: who is kept.  No in-chunk suppression (the common case): every alive candidate.  Otherwise warp 0
            // resolves the chunk; lane l owns candidates l, l + 32, l + 64, l + 96.
            if (!conflict) {
                if (tid < kChunk) {
                    const unsigned a = __ballot_sync(0xffffffffu, S.chunk_alive[tid] != 0);
                    if ((tid & 31) == 0) S.keep_words[tid >> 5] = a;
                }
            } else if (tid < 32) {
                uint32_t alive[kChunkWords], p[kChunkWords][kChunkWords];
#pragma unroll
                for (int c = 0; c < kChunkWords; ++c) alive[c] = __ballot_sync(0xffffffffu, S.chunk_alive[tid + 32 * c] != 0);
#pragma unroll
                for (int c = 0; c < kChunkWords; ++c)
#pragma unroll
                    for (int q = 0; q < kChunkWords; ++q)
                        p[c][q] = q <= c ? (S.chunk_pred[tid + 32 * c][q] & alive[q]) : 0u;
                // Greedy resolution without a serial walk: a candidate is decided as soon as all of its earlier
                // in-chunk suppressors are decided -- kept if none of them was kept, dropped otherwise.  The
                // lowest undecided candidate is always decidable, so this ends; typical chunks need 2-4 rounds.
                uint32_t U[kChunkWords], K[kChunkWords];
#pragma unroll
                for (int c = 0; c < kChunkWords; ++c) { U[c] = alive[c]; K[c] = 0u; }
                for (;;) {
                    uint32_t any_u = 0u;
#pragma unroll
                    for (int c = 0; c < kChunkWords; ++c) any_u |= U[c];
                    if (!any_u) break;
                    uint32_t Rk[kChunkWords], Rs[kChunkWords];
#pragma unroll
                    for (int c = 0; c < kChunkWords; ++c) {
                        const bool in = (U[c] >> tid) & 1u;
                        uint32_t hk = 0u, hu = 0u;
#pragma unroll
                        for (int q = 0; q < kChunkWords; ++q) { hk |= p[c][q] & K[q]; hu |= p[c][q] & U[q]; }
                        Rk[c] = __ballot_sync(0xffffffffu, in && !hk && !hu);
                        Rs[c] = __ballot_sync(0xffffffffu, in && hk);
                    }
#pragma unroll
                    for (int c = 0; c < kChunkWords; ++c) { K[c] |= Rk[c]; U[c] &= ~(Rk[c] | Rs[c]); }
                }
                if (tid == 0) {
#pragma unroll
                    for (int c = 0; c < kChunkWords; ++c) S.keep_words[c] = K[c];
                }
            }
            __syncthreads();
            K2_ACC(11);
            // append the keeps in order; keeps beyond max_det (the lowest-priority ones of the chunk) are dropped
            int added = 0;
            {
                uint32_t kw[kChunkWords];
#pragma unroll
                for (int c = 0; c < kChunkWords; ++c) { kw[c] = S.keep_words[c]; added += __popc(kw[c]); }
                added = min(added, max_det - kept);
                if (tid < kChunk) {
                    const uint32_t mine = S.keep_words[tid >> 5];
                    int before = __popc(mine & ((1u << (tid & 31)) - 1u));
#pragma unroll
                    for (int c = 0; c < kChunkWords; ++c)
                        if (c < (tid >> 5)) before += __popc(kw[c]);
                    const int at = kept + before;
                    if (((mine >> (tid & 31)) & 1u) && at < max_det) {
                        soa_store(kept_box, at, soa_load(chunk_box, tid));
                        if (ARRAY) {
                            aa.keep[at] = static_cast<int32_t>(key_cand<WIDE>(S.keys[c0 + tid]));
                        } else {
                            S.kept_key[at] = S.keys[c0 + tid];
                            S.kept_raw[at] = S.raw[c0 + tid];
                            // (maintained even while the walk tests all pairs: cheap, and the span can only grow)
                            atomicOr(&S.kept_mask[key_cls<WIDE>(S.keys[c0 + tid]) & (kMaskBuckets<KEEP> - 1)][at >> 5], 1u << (at & 31));
                        }
                    }
                    // the chunk's class-bucket mask is all zero again for the next chunk
                    if (!ARRAY && cls_fast && tid < cn) S.chunk_mask[key_cls<WIDE>(S.keys[c0 + tid]) & (kMaskBuckets<KEEP> - 1)][tid >> 5] = 0u;
                }
            }
            kept += added;
            __syncthreads();
            K2_ACC(12);
        }
        K2_STAMP(4);
        K2_ACC_FLUSH();
        processed += n;
        if (kept >= max_det || processed >= limit || processed >= M) break;
        hi_incl = lo - 1;  // lo > 0 here: keys remain below it
    }

    if (ARRAY) {
        if (tid == 0) *aa.keep_cnt = kept;
        return;
    }
    // ---- 5. postprocess_bbox: a kept box survives iff more than one candidate overlaps it by > thr ----------
    if (window) {
        // Every survivor counts, not only the ones the walk visited: they are streamed in blocks of kTranche -- the
        // (single, sorted) tranche still in shared memory when it holds them all, the image's key list otherwise.
        const int warp = tid >> 5, lane = tid & 31;
        // One tranche was walked and the rest of the survivors fits next to it: append them (unordered -- the count filter
        // does not care) instead of streaming and re-decoding the whole list.
        if (!whole && processed == n_tranche && M <= kTranche && !P.topk_sqrt && last_lo > 0) {
            n_tranche = gather_range<THREADS, KEEP>(S, keys, M, smin, 0ull, last_lo - 1, n_tranche);
            whole = n_tranche == M;
        }
        const bool resident = whole;                    // then n_tranche == M and S.keys / S.raw[0..decoded_upto) are valid
        const int total = resident ? min(n_tranche, limit) : M;   // FCOS (top-k) only ever gets here with M <= 300
        for (int r = tid; r < kept; r += THREADS) {
            S.kept_cnt[r] = 0;
#pragma unroll
            for (int q = 0; q < 5; ++q) S.kept_acc[r][q] = 0.0f;
        }
        // x-span of the kept boxes: part of the cross-class disjointness test of every block
        int k_lo = 0x7fffffff, k_hi = static_cast<int>(0x80000000u);
        bool k_fin = true;
        for (int r = tid; r < kept; r += THREADS) {
            const float4 rb = S.kept_raw[r];
            k_fin = k_fin && (fabsf(rb.x) <= 3.0e38f) && (fabsf(rb.z) <= 3.0e38f);
            k_lo = min(k_lo, float_ordered(rb.x));
            k_hi = max(k_hi, float_ordered(rb.z));
        }
        int pf_lo = 0, pf_hi = 0;   // (decode_boxes' span outputs: unused here, the block computes its own below)
        bool pf_bad = false;
        for (int b0 = 0; b0 < total; b0 += kTranche) {
            const int mm = min(kTranche, total - b0);
            __syncthreads();
            if (!resident) {
                for (int i = tid; i < mm; i += THREADS) S.keys[i] = __ldg(keys + b0 + i);
                __syncthreads();
                decode_boxes<false, EXTRA, THREADS, KEEP, T, NHWC, WIDE>(S, P, X, aa, img, 0, mm, pf_lo, pf_hi, pf_bad);
            } else if (decoded_upto < mm) {
                decode_boxes<false, EXTRA, THREADS, KEEP, T, NHWC, WIDE>(S, P, X, aa, img, decoded_upto, mm, pf_lo, pf_hi, pf_bad);
            }
            __syncthreads();
            if (!P.merge_boxes) {
                // offset boxes + areas once per survivor (in place).  The 4096-px class offset keeps boxes of different
                // classes disjoint in x as long as the raw boxes span at most 4095 px: for classes a < b the exact values
                // satisfy x2 + 4096 a < x1' + 4096 b (x2 - x1' <= span < 4096; 4096 cls is exact for every class id), and
                // rounding is monotone, so fl(x2 + 4096 a) <= fl(x1' + 4096 b): the x overlap is <= 0 and the pair cannot
                // reach a positive threshold.  This needs no bound on the offset values, so it holds where they pass 2^23
                // (class 2047 plus a box coordinate) and the float32 spacing grows to 1.  Then a kept box only needs the
                // survivors of its own class: bucket the block by class (counting sort of indices in shared memory, up to
                // kBins / 2 = 1024 classes; wider plans test every pair) and walk one bucket per kept box.  Otherwise
                // (huge boxes -- the reference then lets classes interact) every pair is tested.
                int lo_x = k_lo, hi_x = k_hi;
                bool finite = k_fin;
                for (int jj = tid; jj < mm; jj += THREADS) {
                    const uint64_t key = S.keys[jj];
                    const float off = P.class_aware ? __fmul_rn(static_cast<float>(key_cls<WIDE>(key)), 4096.0f) : 0.0f;
                    const float4 rb = S.raw[jj];
                    finite = finite && (fabsf(rb.x) <= 3.0e38f) && (fabsf(rb.z) <= 3.0e38f);  // false for NaN / inf
                    lo_x = min(lo_x, float_ordered(rb.x));
                    hi_x = max(hi_x, float_ordered(rb.z));
                    const OffBox b = make_offbox(rb, off);
                    S.raw[jj] = make_float4(b.x1, b.y1, b.x2, b.y2);
                    S.area[jj] = b.area;
                }
                lo_x = __reduce_min_sync(0xffffffffu, lo_x);
                hi_x = __reduce_max_sync(0xffffffffu, hi_x);
                if (tid == 0) { S.span_lo = 0x7fffffff; S.span_hi = static_cast<int>(0x80000000u); }
                const bool all_finite = __syncthreads_and(finite ? 1 : 0);
                if (lane == 0) { atomicMin(&S.span_lo, lo_x); atomicMax(&S.span_hi, hi_x); }
                __syncthreads();
                const float span = __fsub_rn(ordered_float(S.span_hi), ordered_float(S.span_lo));
                const bool buckets = P.class_aware && thr.positive && P.C <= kBins / 2 && all_finite && span <= 4095.0f;
                if (buckets) {
                    uint32_t *cnt_cls = S.hist;               // [0, C): bucket starts; [kBins/2, kBins/2 + C): fill cursors
                    uint32_t *cursor = S.hist + kBins / 2;
                    for (int c = tid; c < kBins / 2; c += THREADS) cnt_cls[c] = 0;
                    __syncthreads();
                    for (int jj = tid; jj < mm; jj += THREADS) atomicAdd(&cnt_cls[key_cls<WIDE>(S.keys[jj])], 1u);
                    __syncthreads();
                    // exclusive scan over the classes: PERC consecutive classes per thread
                    constexpr int PERC = (kBins / 2) / THREADS;
                    uint32_t mine[PERC];
                    uint32_t part = 0;
#pragma unroll
                    for (int q = 0; q < PERC; ++q) { mine[q] = cnt_cls[PERC * tid + q]; part += mine[q]; }
                    uint32_t incl = part;
#pragma unroll
                    for (int d = 1; d < 32; d <<= 1) {
                        const uint32_t v = __shfl_up_sync(0xffffffffu, incl, d);
                        if (lane >= d) incl += v;
                    }
                    if (lane == 31) S.warp_tmp[warp] = incl;
                    __syncthreads();
                    if (warp == 0) {
                        uint32_t w = lane < THREADS / 32 ? S.warp_tmp[lane] : 0u;
#pragma unroll
                        for (int d = 1; d < 32; d <<= 1) {
                            const uint32_t v = __shfl_up_sync(0xffffffffu, w, d);
                            if (lane >= d) w += v;
                        }
                        S.warp_tmp[lane] = w;  // inclusive over warps
                    }
                    __syncthreads();
                    uint32_t start = incl - part + (warp > 0 ? S.warp_tmp[warp - 1] : 0u);
#pragma unroll
                    for (int q = 0; q < PERC; ++q) {
                        cnt_cls[PERC * tid + q] = start;
                        cursor[PERC * tid + q] = start;
                        start += mine[q];
                    }
                    __syncthreads();
                    for (int jj = tid; jj < mm; jj += THREADS) {
                        const uint32_t at = atomicAdd(&cursor[key_cls<WIDE>(S.keys[jj])], 1u);
                        S.order[at] = static_cast<uint16_t>(jj);
                    }
                    __syncthreads();
                    for (int r = warp; r < kept; r += THREADS / 32) {
                        const OffBox br = soa_load(kept_box, r);
                        const uint32_t cls_r = key_cls<WIDE>(S.kept_key[r]);
                        const int lo = static_cast<int>(cnt_cls[cls_r]), hi = static_cast<int>(cursor[cls_r]);
                        int c = 0;
                        for (int q = lo + lane; q < hi; q += 32) {
                            const int jj = S.order[q];
                            const float4 o = S.raw[jj];
                            const float dw = __fsub_rn(fminf(br.x2, o.z), fmaxf(br.x1, o.x));
                            const float dh = __fsub_rn(fminf(br.y2, o.w), fmaxf(br.y1, o.y));
                            if (!(dw > 0.0f && dh > 0.0f)) continue;
                            c += iou_decide<true>(dw, dh, br.area, S.area[jj], thr) ? 1 : 0;
                        }
                        c = __reduce_add_sync(0xffffffffu, c);
                        if (lane == 0) S.kept_cnt[r] = static_cast<uint16_t>(S.kept_cnt[r] + c);
                    }
                } else {
                    for (int r = warp; r < kept; r += THREADS / 32) {
                        const OffBox br = soa_load(kept_box, r);
                        int c = 0;
                        for (int jj = lane; jj < mm; jj += 32) {
                            const float4 o = S.raw[jj];  // offset box (x1, y1, x2, y2)
                            const float dw = __fsub_rn(fminf(br.x2, o.z), fmaxf(br.x1, o.x));
                            const float dh = __fsub_rn(fminf(br.y2, o.w), fmaxf(br.y1, o.y));
                            if (thr.positive && !(dw > 0.0f && dh > 0.0f)) continue;
                            c += iou_decide<true>(dw, dh, br.area, S.area[jj], thr) ? 1 : 0;
                        }
                        c = __reduce_add_sync(0xffffffffu, c);
                        if (lane == 0) S.kept_cnt[r] = static_cast<uint16_t>(S.kept_cnt[r] + c);
                    }
                }
            } else {
                for (int r = warp; r < kept; r += THREADS / 32) {
                    const OffBox br = soa_load(kept_box, r);
                    int c = 0;
                    float ax = 0.f, ay = 0.f, az = 0.f, aw = 0.f, ws = 0.f;
                    for (int jj = lane; jj < mm; jj += 32) {
                        const uint64_t key = S.keys[jj];
                        const float off = P.class_aware ? __fmul_rn(static_cast<float>(key_cls<WIDE>(key)), 4096.0f) : 0.0f;
                        const float4 rj = S.raw[jj];
                        if (iou_reaches<true>(br, make_offbox(rj, off), thr)) {
                            ++c;
                            // trainer/eval_retinanet.py:346-349 (float32 weights, float32 dot)
                            const float w = key_score(key);
                            ax = __fadd_rn(ax, __fmul_rn(w, rj.x));
                            ay = __fadd_rn(ay, __fmul_rn(w, rj.y));
                            az = __fadd_rn(az, __fmul_rn(w, rj.z));
                            aw = __fadd_rn(aw, __fmul_rn(w, rj.w));
                            ws = __fadd_rn(ws, w);
                        }
                    }
                    c = __reduce_add_sync(0xffffffffu, c);
#pragma unroll
                    for (int d = 16; d > 0; d >>= 1) {
                        ax = __fadd_rn(ax, __shfl_xor_sync(0xffffffffu, ax, d));
                        ay = __fadd_rn(ay, __shfl_xor_sync(0xffffffffu, ay, d));
                        az = __fadd_rn(az, __shfl_xor_sync(0xffffffffu, az, d));
                        aw = __fadd_rn(aw, __shfl_xor_sync(0xffffffffu, aw, d));
                        ws = __fadd_rn(ws, __shfl_xor_sync(0xffffffffu, ws, d));
                    }
                    if (lane == 0) {
                        S.kept_cnt[r] = static_cast<uint16_t>(S.kept_cnt[r] + c);
                        S.kept_acc[r][0] = __fadd_rn(S.kept_acc[r][0], ax);
                        S.kept_acc[r][1] = __fadd_rn(S.kept_acc[r][1], ay);
                        S.kept_acc[r][2] = __fadd_rn(S.kept_acc[r][2], az);
                        S.kept_acc[r][3] = __fadd_rn(S.kept_acc[r][3], aw);
                        S.kept_acc[r][4] = __fadd_rn(S.kept_acc[r][4], ws);
                    }
                }
            }
        }
        __syncthreads();
        for (int r = tid; r < kept; r += THREADS) {
            S.kept_flag[r] = S.kept_cnt[r] > 1;
            if (P.merge_boxes) {
                const float den = __fadd_rn(S.kept_acc[r][4], 1e-16f);
                S.kept_raw[r] = make_float4(__fdiv_rn(S.kept_acc[r][0], den), __fdiv_rn(S.kept_acc[r][1], den),
                                            __fdiv_rn(S.kept_acc[r][2], den), __fdiv_rn(S.kept_acc[r][3], den));
            }
        }
    } else {
        for (int r = tid; r < kept; r += THREADS) S.kept_flag[r] = 1;
    }
    __syncthreads();
    K2_STAMP(5);
    // ---- ordered write of the surviving rows ---------------------------------------------------------------
    // optional letterbox undo (val_yolov5.py:166-172) on the way out: the filters above saw the un-mapped boxes
    float lb_scale = 1.0f, lb_top = 0.0f, lb_left = 0.0f, lb_hi_y = 0.0f, lb_hi_x = 0.0f;
    const bool lb = !ARRAY && P.letterbox != nullptr;
    if (lb) {
        const float *t = P.letterbox + static_cast<size_t>(img) * 5;
        lb_scale = __ldg(t);
        lb_top = __ldg(t + 1);
        lb_left = __ldg(t + 2);
        lb_hi_y = __fsub_rn(__ldg(t + 3), 1.0f);
        lb_hi_x = __fsub_rn(__ldg(t + 4), 1.0f);
    }
    // Rows are first laid out in shared memory (the tranche's box array is free by now), then copied out with full-width
    // contiguous stores -- to the caller's buffer or, in a detection gather, to every rank's receive slot.  (Storing the
    // six floats of a row one by one cost 6 partial-sector writes per row and destination: over NVLink, with 8
    // destinations, that tripled the kernel's time.)
    float *stage = reinterpret_cast<float *>(S.raw);   // kTranche * 16 B >= max_det (<= 1024) * 24 B
    int written = 0;
    for (int r0 = 0; r0 < kept; r0 += THREADS) {
        const int r = r0 + tid;
        bool pass = false;
        float4 box = make_float4(0.f, 0.f, 0.f, 0.f);
        uint64_t key = 0;
        if (r < kept) {
            box = S.kept_raw[r];
            key = S.kept_key[r];
            pass = S.kept_flag[r] != 0;
            if (pass && P.small_box_filter)  // remove_small_boxes, trainer/eval_yolov7.py:203-213
                pass = (__fsub_rn(box.z, box.x) > P.min_box_wh) && (__fsub_rn(box.w, box.y) > P.min_box_wh);
        }
        const unsigned bal = __ballot_sync(0xffffffffu, pass);
        __syncthreads();   // warp_tmp of the previous round has been read
        if ((tid & 31) == 0) S.warp_tmp[tid >> 5] = __popc(bal);
        __syncthreads();
        int before = written, total = written;
        for (int w = 0; w < THREADS / 32; ++w) {
            const int c = static_cast<int>(S.warp_tmp[w]);
            if (w < (tid >> 5)) before += c;
            total += c;
        }
        if (pass) {
            const int at = before + __popc(bal & ((1u << (tid & 31)) - 1u));
            const float sc = key_score(key);
            const float s_out = P.topk_sqrt ? sqrtf(sc) : sc;  // FCOS: x[:, 4] = sqrt(x[:, 4]) (trainer/eval_fcos.py:281)
            const float c_out = static_cast<float>(key_cls<WIDE>(key));
            if (lb) {
                box.x = fminf(fmaxf(__fdiv_rn(__fsub_rn(box.x, lb_left), lb_scale), 1.0f), lb_hi_x);
                box.z = fminf(fmaxf(__fdiv_rn(__fsub_rn(box.z, lb_left), lb_scale), 1.0f), lb_hi_x);
                box.y = fminf(fmaxf(__fdiv_rn(__fsub_rn(box.y, lb_top), lb_scale), 1.0f), lb_hi_y);
                box.w = fminf(fmaxf(__fdiv_rn(__fsub_rn(box.w, lb_top), lb_scale), 1.0f), lb_hi_y);
            }
            float *row = stage + at * 6;
            row[0] = box.x; row[1] = box.y; row[2] = box.z; row[3] = box.w;
            row[4] = s_out;
            row[5] = c_out;
            if (det_idx) det_idx[static_cast<size_t>(img) * max_det + at] = static_cast<int32_t>(key_cand<WIDE>(key));
        }
        written = total;
    }
    {
        const int nfl = written * 6;
        const int nfl4 = (nfl + 3) & ~3;
        if (tid < nfl4 - nfl) stage[nfl + tid] = 0.0f;   // the last 16-byte store may reach past the rows: defined bytes
        // detection gather: every peer must have consumed the previous use of this slot (its ack, published at the start
        // of its current step, arrived long ago in the steady state) before anything is stored into its region
        if (G.world > 0 && tid < G.world && tid != G.rank && !spin_until_reached(G.my_ack + tid, *G.use)) atomicExch(G.err, 1u);
        __syncthreads();
        const size_t img_off = static_cast<size_t>(img) * max_det * 6;
        const int ndst = G.world > 0 ? G.world : 1;
        // a 16-byte store needs an even max_det (image rows start on 16-byte boundaries) and must stay inside the image
        const bool wide = (max_det & 1) == 0;
        for (int d = 0; d < ndst; ++d) {
            float *dst = (G.world > 0 ? G.rows[d] : dets) + img_off;
            if (wide && (reinterpret_cast<uintptr_t>(dst) & 15u) == 0) {
                for (int e = tid; e < nfl4 / 4; e += THREADS)
                    reinterpret_cast<float4 *>(dst)[e] = reinterpret_cast<const float4 *>(stage)[e];
            } else {
                for (int e = tid; e < nfl / 2; e += THREADS)   // rows are 24 bytes: always 8-byte aligned
                    reinterpret_cast<float2 *>(dst)[e] = reinterpret_cast<const float2 *>(stage)[e];
            }
        }
    }
    K2_STAMP(6);
    if (tid == 0) {
        const int value = (written == 0 && P.none_when_empty) ? -1 : written;
        if (G.world > 0) {
            for (int d = 0; d < G.world; ++d) G.cnt[d][img] = value;
        } else {
            det_cnt[img] = value;
        }
    }
    if (G.world > 0) {
        // release: every row / count store of this CTA is ordered before the arrival count each peer will see
        __threadfence_system();
        __syncthreads();
        if (tid < G.world) atomicAdd_system(G.arrived[tid], 1u);
    }
}

// ---- host side ---------------------------------------------------------------------------------------------------------
// CTA flavour (launch_any): 512 or 1024 threads.  Profiling builds can force it (ysb_debug_set_nms_threads).
static int g_force_threads = 0;
void debug_set_nms_threads(int t) { g_force_threads = t; }
#ifdef YSB_PROFILING_VARIANTS
// profiling build only: YSB_NMS_THREADS=512|1024 forces the CTA flavour (read once)
static int env_force_threads()
{
    static int v = -1;
    if (v < 0) {
        const char *e = getenv("YSB_NMS_THREADS");
        v = e ? atoi(e) : 0;
    }
    return v;
}
#endif

static int device_sm_count()
{
    int dev = 0, n = 148;
    if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    return n;
}

template <typename EXTRA, int THREADS, int KEEP, typename T, bool NHWC, bool WIDE>
static cudaError_t launch_flavour(const Plan &P, const EXTRA &X, const uint64_t *d_keys, int64_t key_cap, const int32_t *d_counts,
                                  float *d_dets, int32_t *d_det_idx, int32_t *d_det_cnt, cudaStream_t stream, const GatherSink &G)
{
    // per-device attribute; set on every launch (host-side, sub-microsecond) so that a process driving several
    // devices never launches with the default 48 KB limit
    auto kern = k_select_nms<false, EXTRA, THREADS, KEEP, T, NHWC, WIDE>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(sizeof(NmsSmem<KEEP>)));
    if (e != cudaSuccess) return e;
    ArrayArgs aa{};
    size_t smem = sizeof(NmsSmem<KEEP>);
#ifdef YSB_PROFILING_VARIANTS
    {   // profiling build only: YSB_NMS_SMEM=<bytes> requests more shared memory (limits the CTAs per SM)
        static long pad = -1;
        if (pad < 0) { const char *e = getenv("YSB_NMS_SMEM"); pad = e ? atol(e) : 0; }
        if (static_cast<size_t>(pad) > smem) {
            smem = static_cast<size_t>(pad);
            e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
            if (e != cudaSuccess) return e;
        }
    }
#endif
    kern<<<P.batch, THREADS, smem, stream>>>(P, X, d_keys, key_cap, d_counts, d_dets, d_det_idx, d_det_cnt, aa, G);
    return cudaGetLastError();
}

template <typename EXTRA, typename T, bool NHWC, bool WIDE>
static cudaError_t launch_any(const Plan &P, const EXTRA &X, const uint64_t *d_keys, int64_t key_cap, const int32_t *d_counts,
                              float *d_dets, int32_t *d_det_idx, int32_t *d_det_cnt, cudaStream_t stream, const GatherSink *sink)
{
    if (P.batch == 0) return cudaSuccess;
    GatherSink G;
    if (sink) G = *sink;
    else memset(&G, 0, sizeof(G));
    const bool small_keep = P.max_det <= 320;
    // 512 threads: the CTA leaves half of its SM's registers to three filter CTAs of the batches that follow, and two of
    // them fit an SM when there are more images than SMs.  1024 threads: lowest latency per image -- small batches, the
    // YOLOv8 DFL box decode (THREADS / 4 boxes per DRAM round trip) and very long key lists, whose selection passes
    // scale with M / THREADS.  Measured on B200, 4 batches in flight, images/s 1024 -> 512 threads: YOLOv5s b=64 674 k ->
    // 738 k, YOLOv7 b=64 584 k -> 623 k, b=8 451 k -> 397 k, YOLOv8 b=64 452 k -> 442 k, RetinaNet (76 725) 208 k -> 204 k.
    const bool dfl = P.family == YSB_YOLOV8 && P.input_kind == YSB_INPUT_RAW_HEADS;
    int threads = 1024;
    if (small_keep && (P.batch > device_sm_count() || (P.batch >= 32 && !dfl && P.N <= 32768))) threads = 512;
#ifdef YSB_PROFILING_VARIANTS
    if (env_force_threads()) g_force_threads = env_force_threads();
#endif
    if (g_force_threads == 512 && small_keep) threads = 512;
    if (g_force_threads == 1024) threads = 1024;
    if (!small_keep) return launch_flavour<EXTRA, 1024, 1024, T, NHWC, WIDE>(P, X, d_keys, key_cap, d_counts, d_dets, d_det_idx, d_det_cnt, stream, G);
    if (threads == 512) return launch_flavour<EXTRA, 512, 320, T, NHWC, WIDE>(P, X, d_keys, key_cap, d_counts, d_dets, d_det_idx, d_det_cnt, stream, G);
    return launch_flavour<EXTRA, 1024, 320, T, NHWC, WIDE>(P, X, d_keys, key_cap, d_counts, d_dets, d_det_idx, d_det_cnt, stream, G);
}

template <typename EXTRA, bool NHWC, bool WIDE>
static cudaError_t launch_any_dt(const Plan &P, const EXTRA &X, const uint64_t *d_keys, int64_t key_cap, const int32_t *d_counts,
                                 float *d_dets, int32_t *d_det_idx, int32_t *d_det_cnt, cudaStream_t stream,
                                 const GatherSink *sink, int dtype)
{
    switch (dtype) {
    case YSB_F16: return launch_any<EXTRA, __half, NHWC, WIDE>(P, X, d_keys, key_cap, d_counts, d_dets, d_det_idx, d_det_cnt, stream, sink);
    case YSB_BF16:
        return launch_any<EXTRA, __nv_bfloat16, NHWC, WIDE>(P, X, d_keys, key_cap, d_counts, d_dets, d_det_idx, d_det_cnt, stream, sink);
    default: return launch_any<EXTRA, float, NHWC, WIDE>(P, X, d_keys, key_cap, d_counts, d_dets, d_det_idx, d_det_cnt, stream, sink);
    }
}

// NHWC heads (LAYOUT_ROWS_NHWC, YSB_INPUT_RAW_HEADS_NHWC): the kernel's box decode addresses channels-last memory.
// More than 1024 classes: wide sort keys (never with NHWC heads, whose rows that wide the ABI refuses).
template <typename EXTRA>
static cudaError_t launch_any_layout(const Plan &P, const EXTRA &X, const uint64_t *d_keys, int64_t key_cap,
                                     const int32_t *d_counts, float *d_dets, int32_t *d_det_idx, int32_t *d_det_cnt,
                                     cudaStream_t stream, const GatherSink *sink, int dtype)
{
    if (P.layout == LAYOUT_ROWS_NHWC) return launch_any_dt<EXTRA, true, false>(P, X, d_keys, key_cap, d_counts, d_dets, d_det_idx, d_det_cnt, stream, sink, dtype);
    if (wide_keys(P.C)) return launch_any_dt<EXTRA, false, true>(P, X, d_keys, key_cap, d_counts, d_dets, d_det_idx, d_det_cnt, stream, sink, dtype);
    return launch_any_dt<EXTRA, false, false>(P, X, d_keys, key_cap, d_counts, d_dets, d_det_idx, d_det_cnt, stream, sink, dtype);
}

cudaError_t launch_select_nms(const Plan &P, const uint64_t *d_keys, int64_t key_cap, const int32_t *d_counts,
                              float *d_dets, int32_t *d_det_idx, int32_t *d_det_cnt, cudaStream_t stream,
                              const GatherSink *sink, int dtype)
{
    return launch_any_layout(P, NoExtraPasses{}, d_keys, key_cap, d_counts, d_dets, d_det_idx, d_det_cnt, stream, sink, dtype);
}

// test-time augmentation: one selection/NMS over the key lists the passes appended to; X describes passes 1..n.  sink:
// as launch_select_nms (nullptr = the caller's dets / det_cnt; a detection gather = every rank's slot)
cudaError_t launch_select_nms_tta(const Plan &P, const ExtraPasses &X, const uint64_t *d_keys, int64_t key_cap,
                                  const int32_t *d_counts, float *d_dets, int32_t *d_det_idx, int32_t *d_det_cnt,
                                  cudaStream_t stream, const GatherSink *sink, int dtype)
{
    return launch_any_layout(P, X, d_keys, key_cap, d_counts, d_dets, d_det_idx, d_det_cnt, stream, sink, dtype);
}

// ---- array flavour: utils.numba_nms / utils.gpu_nms over one explicit (m,4)/(m) pair ---------------------------
// zero scores are never kept (utils/nms.py:16 "while score.sum() > 0"); keys carry the array index.
__global__ void k_array_keys(const float *__restrict__ scores, int m, uint64_t *__restrict__ keys, int32_t *__restrict__ counts)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const bool ok = i < m && scores[i] > 0.0f;
    const unsigned bal = __ballot_sync(0xffffffffu, ok);
    if (!bal) return;
    const unsigned lane = threadIdx.x & 31u;
    const uint32_t sb = ok ? __float_as_uint(scores[i]) : 0u;
    const uint32_t wmax = __reduce_max_sync(0xffffffffu, sb);
    const uint32_t wmin = __reduce_max_sync(0xffffffffu, ok ? ~sb : 0u);
    int base = 0;
    if (lane == 0) {
        base = atomicAdd(counts, __popc(bal));
        atomicMax(reinterpret_cast<unsigned int *>(counts + 2), wmax);
        atomicMax(reinterpret_cast<unsigned int *>(counts + 3), wmin);
    }
    base = __shfl_sync(0xffffffffu, base, 0);
    if (ok) keys[base + __popc(bal & ((1u << lane) - 1u))] = pack_key(scores[i], static_cast<uint32_t>(i), 0u);
}

static size_t align256(size_t x) { return (x + 255) & ~static_cast<size_t>(255); }

size_t array_nms_workspace_bytes(int64_t m)
{
    const size_t mm = static_cast<size_t>(m > 0 ? m : 1);
    return align256(sizeof(uint64_t) * mm) + 3 * align256(sizeof(float2) * mm) + align256(sizeof(int32_t) * 4) + 256;
}

cudaError_t launch_array_nms(const float *d_boxes, const float *d_scores, int64_t m, double iou_thr, int cmp, int iou_kind,
                             int64_t max_keep, void *ws, int32_t *d_keep, int32_t *d_keep_cnt, cudaStream_t stream)
{
    if (m == 0) return cudaMemsetAsync(d_keep_cnt, 0, sizeof(int32_t), stream);
    const size_t mm = static_cast<size_t>(m);
    uintptr_t base = (reinterpret_cast<uintptr_t>(ws) + 255) & ~static_cast<uintptr_t>(255);
    uint64_t *keys = reinterpret_cast<uint64_t *>(base);
    const size_t seg = align256(sizeof(float2) * mm);
    uintptr_t kb = base + align256(sizeof(uint64_t) * mm);
    BoxSoA kept{reinterpret_cast<float2 *>(kb), reinterpret_cast<float2 *>(kb + seg), reinterpret_cast<float *>(kb + 2 * seg)};
    int32_t *counts = reinterpret_cast<int32_t *>(kb + 3 * seg);
    cudaError_t e = cudaMemsetAsync(counts, 0, sizeof(int32_t) * 4, stream);
    if (e != cudaSuccess) return e;
    k_array_keys<<<static_cast<unsigned>((m + 255) / 256), 256, 0, stream>>>(d_scores, static_cast<int>(m), keys, counts);
    // the kept list of the array flavour lives in the global workspace: the shared-memory kept arrays stay minimal
    auto kern = k_select_nms<true, NoExtraPasses, 1024, 64>;
    e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(sizeof(NmsSmem<64>)));
    if (e != cudaSuccess) return e;
    Plan P;
    memset(&P, 0, sizeof(P));
    P.batch = 1;
    P.N = static_cast<int>(m);
    P.iou_thr = iou_thr;
    P.max_det = static_cast<int>((max_keep > 0 && max_keep < m) ? max_keep : m);
    ArrayArgs aa;
    aa.boxes = reinterpret_cast<const float4 *>(d_boxes);
    aa.kept = kept;
    aa.keep = d_keep;
    aa.keep_cnt = d_keep_cnt;
    aa.iou_kind = iou_kind;
    aa.cmp = cmp;
    aa.thr32 = static_cast<float>(iou_thr);
    GatherSink G;
    memset(&G, 0, sizeof(G));
    kern<<<1, 1024, sizeof(NmsSmem<64>), stream>>>(P, NoExtraPasses{}, keys, m, counts, nullptr, nullptr, nullptr, aa, G);
    return cudaGetLastError();
}

#ifdef YSB_K2_TIMING
cudaError_t debug_k2_timing(long long *host_out) { return cudaMemcpyFromSymbol(host_out, g_k2_timing, sizeof(g_k2_timing)); }
#endif

}  // namespace ysb
