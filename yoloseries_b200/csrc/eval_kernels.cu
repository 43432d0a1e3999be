// eval_kernels.cu -- the consumers right after the kept rows (SURVEY.md 8f "next" rows):
//   * mAP_v2.compute_tp and its pairwise IoU        utils/mAP.py:18-42, 70-100   (k_compute_tp, k_map_iou; k_match_tp
//                                                   and k_match_compact on the post-processors' own row blocks)
//   * weighted-box-fusion                           utils/weighted_fusion_bbox.py:41-96, trainer/eval_yolov5.py:44-92
//                                                   (k_wbf)
// Small, latency-bound problems (<= max_det predictions x a few dozen ground-truth boxes per image; a few thousand boxes
// per image for the fusion): one CTA per image / per (image, label) segment, everything else is parallel over images.
#include "ysb_internal.cuh"

#include <climits>

namespace ysb {

// ---- utils/mAP.py:18-42 ------------------------------------------------------------------------------------------------
// numpy, in the arrays' own precision T: areas = w*h, inter = max(0, .) * max(0, .), iou = inter / clip(a1 + a2 - inter,
// 1e-6, 1e7).  a = ground truth row (x1, y1, x2, y2, ...), b = prediction row.
// B: element type of b's storage, widened exactly to T on load (float32 rows against float64 ground truth).
template <typename T, typename B = T>
__device__ __forceinline__ T map_iou(const T *a, const B *b)
{
    const T a1 = (a[2] - a[0]) * (a[3] - a[1]);
    const T a2 = (T(b[2]) - T(b[0])) * (T(b[3]) - T(b[1]));
    const T xmin = a[0] > T(b[0]) ? a[0] : T(b[0]), ymin = a[1] > T(b[1]) ? a[1] : T(b[1]);   // np.maximum / np.minimum
    const T xmax = a[2] < T(b[2]) ? a[2] : T(b[2]), ymax = a[3] < T(b[3]) ? a[3] : T(b[3]);
    T w = xmax - xmin, h = ymax - ymin;
    w = w > T(0) ? w : T(0);
    h = h > T(0) ? h : T(0);
    const T inter = w * h;
    T den = (a1 + a2) - inter;
    den = den < T(1e-6) ? T(1e-6) : (den > T(10000000) ? T(10000000) : den);
    return inter / den;
}

template <typename T>
__global__ void __launch_bounds__(256) k_map_iou(const T *__restrict__ b1, int64_t n, int w1, const T *__restrict__ b2,
                                                 int64_t m, int w2, T *__restrict__ out)
{
    const int64_t i = blockIdx.y;
    const int64_t j = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= n || j >= m) return;
    out[i * m + j] = map_iou<T>(b1 + i * w1, b2 + j * w2);
}

struct TpThresholds {
    double v[10];
};

// The best ground-truth box of prediction j under the reference's ordering (utils/mAP.py:88-96): pairs with
// iou >= thr[0] and equal label, sorted by IoU descending; np.unique(pred) keeps the first pair of every prediction.
// Equal IoUs: argsort()[::-1] of a stable sort visits the LATER pair first, i.e. the larger ground-truth index.
// P: element type of the prediction rows (T, or float32 rows widened to float64).
template <typename T, typename P>
__device__ __forceinline__ int best_gt(const T *gt, int n, const P *p, double thr0, T &best_iou)
{
    int bi = -1;
    T bv = T(0);
    for (int i = 0; i < n; ++i) {
        const T *g = gt + static_cast<int64_t>(i) * 5;
        const T v = map_iou<T, P>(g, p);
        if (static_cast<double>(v) >= thr0 && g[4] == static_cast<T>(p[5]) && (bi < 0 || v >= bv)) {
            bi = i;
            bv = v;
        }
    }
    best_iou = bv;
    return bi;
}

// The matching of one image, run by one CTA.  Its n ground-truth rows (x1, y1, x2, y2, cls) are gt[g0 ..], its m kept
// rows (x1, y1, x2, y2, score, cls) pred[p0 ..], its tp rows (10 bytes) tp[t0 ..]; first_pred[g0 ..]: one int per
// ground-truth row (workspace).
//   phase 1: every prediction finds its best ground-truth box and bids for it with atomicMin(pred index): the second
//            np.unique (over the ground-truth column of the pred-ordered list) keeps the LOWEST prediction index of
//            every ground-truth box -- not the highest IoU; that is the reference's behaviour and it is kept.
//   phase 2: the winning prediction of every ground-truth box gets tp[j, t] = iou >= thr[t] (float64 comparison).
// The kernels below differ only in where an image's rows live (the addressing); all of them match through this body.
template <typename T, typename P>
__device__ __forceinline__ void match_image(const T *__restrict__ gt, int64_t g0, int n, const P *__restrict__ pred,
                                            int64_t p0, int m, const TpThresholds &thr, int32_t *__restrict__ first_pred,
                                            uint8_t *__restrict__ tp, int64_t t0)
{
    for (int i = threadIdx.x; i < n; i += blockDim.x) first_pred[g0 + i] = INT_MAX;
    for (int e = threadIdx.x; e < m * 10; e += blockDim.x) tp[t0 * 10 + e] = 0;
    __syncthreads();
    const T *g = gt + g0 * 5;
    for (int j = threadIdx.x; j < m; j += blockDim.x) {
        T v;
        const int bi = best_gt<T, P>(g, n, pred + (p0 + j) * 6, thr.v[0], v);
        if (bi >= 0) atomicMin(first_pred + g0 + bi, j);
    }
    __syncthreads();
    for (int j = threadIdx.x; j < m; j += blockDim.x) {
        T v;
        const int bi = best_gt<T, P>(g, n, pred + (p0 + j) * 6, thr.v[0], v);
        if (bi >= 0 && first_pred[g0 + bi] == j) {
#pragma unroll
            for (int t = 0; t < 10; ++t) tp[(t0 + j) * 10 + t] = static_cast<double>(v) >= thr.v[t] ? 1 : 0;
        }
    }
}

// ysb_compute_tp: one CTA per image; images are concatenated, gt_off / pred_off (batch + 1) are row offsets.
template <typename T>
__global__ void __launch_bounds__(256) k_compute_tp(const T *__restrict__ gt, const int64_t *__restrict__ gt_off,
                                                    const T *__restrict__ pred, const int64_t *__restrict__ pred_off,
                                                    const __grid_constant__ TpThresholds thr, int32_t *__restrict__ first_pred,
                                                    uint8_t *__restrict__ tp)
{
    const int img = blockIdx.x;
    const int64_t g0 = gt_off[img], p0 = pred_off[img];
    const int n = static_cast<int>(gt_off[img + 1] - g0), m = static_cast<int>(pred_off[img + 1] - p0);
    match_image<T, T>(gt, g0, n, pred, p0, m, thr, first_pred, tp, p0);
}

// ---- matching in the post-processors' own layouts (ysb_match_tp, ysb_match_compact) ---------------------------------
// Image k = rank * batch + i of a step.  Rows and counts of a rank start rows_rank_bytes / cnt_rank_bytes after those
// of the previous one (the 256-byte padded regions of a gather slot); ground truth and its counts are dense.
__device__ __forceinline__ int step_count(const ysb_match_step &s, int k)
{
    const int r = k / s.batch, i = k - r * s.batch;
    return reinterpret_cast<const int32_t *>(reinterpret_cast<const unsigned char *>(s.d_cnt) + r * s.cnt_rank_bytes)[i];
}

__device__ __forceinline__ const float *step_rows(const ysb_match_step &s, int k)
{
    const int r = k / s.batch, i = k - r * s.batch;
    return reinterpret_cast<const float *>(reinterpret_cast<const unsigned char *>(s.d_rows) + r * s.rows_rank_bytes) +
           static_cast<int64_t>(i) * s.max_det * 6;
}

// rows of image k that take part (a count of -1 -- the reference's None -- has none; absent images are not asked)
__device__ __forceinline__ int step_preds(const ysb_match_step &s, int c) { return c < 0 ? 0 : (c < s.max_det ? c : s.max_det); }

__device__ __forceinline__ int step_targets(const ysb_match_step &s, int k)
{
    const int n = s.d_gt_cnt[k];
    return n < 0 ? 0 : (n < s.max_gt ? n : s.max_gt);
}

// One CTA per image of the step; absent images (YSB_CNT_ABSENT) keep their tp rows.  Rows are float32 and are widened
// to T (the ground truth's type) on load, as ysb_compute_tp matches float32 rows promoted to float64.
template <typename T>
__global__ void __launch_bounds__(256) k_match_tp(const __grid_constant__ ysb_match_step s,
                                                  const __grid_constant__ TpThresholds thr, int32_t *__restrict__ first_pred,
                                                  uint8_t *__restrict__ tp)
{
    const int k = blockIdx.x;
    const int c = step_count(s, k);
    if (c == YSB_CNT_ABSENT) return;
    match_image<T, float>(static_cast<const T *>(s.d_gt), static_cast<int64_t>(k) * s.max_gt, step_targets(s, k),
                          step_rows(s, k), 0, step_preds(s, c), thr, first_pred, tp, static_cast<int64_t>(k) * s.max_det);
}

// The sum over the CTA of one value per thread (blockDim.x a multiple of 32, <= 1024).
__device__ __forceinline__ long long block_sum(long long v, long long *red)
{
    for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
    __syncthreads();
    long long t = 0;
    for (int w = 0; w < static_cast<int>(blockDim.x >> 5); ++w) t += red[w];
    __syncthreads();
    return t;
}

// One CTA per image of the step: its place among the step's present images (a prefix sum over the counts before it),
// then a scatter of its kept rows' score, class and tp row and of its targets' classes after what earlier steps
// appended (acc_in = {rows, targets} so far).  The last CTA writes acc_in + the step's totals to acc_out.  Writes beyond
// the capacities are dropped; the totals still count them.
template <typename T>
__global__ void __launch_bounds__(256) k_match_compact(const __grid_constant__ ysb_match_step s, const uint8_t *__restrict__ tp,
                                                       const long long *__restrict__ acc_in, long long *__restrict__ acc_out,
                                                       float *__restrict__ conf, float *__restrict__ pred_cls,
                                                       uint8_t *__restrict__ tp_out, long long row_cap,
                                                       double *__restrict__ target_cls, long long target_cap)
{
    __shared__ long long red[2][32];
    const int k = blockIdx.x;
    long long rows = 0, tgts = 0;
    for (int q = threadIdx.x; q < k; q += blockDim.x) {
        const int c = step_count(s, q);
        if (c == YSB_CNT_ABSENT) continue;
        rows += step_preds(s, c);
        tgts += step_targets(s, q);
    }
    rows = block_sum(rows, red[0]);
    tgts = block_sum(tgts, red[1]);
    const int c = step_count(s, k);
    const bool present = c != YSB_CNT_ABSENT;
    const int m = present ? step_preds(s, c) : 0, n = present ? step_targets(s, k) : 0;
    const long long r0 = acc_in[0] + rows, g0 = acc_in[1] + tgts;
    if (k == static_cast<int>(gridDim.x) - 1 && threadIdx.x == 0) {
        acc_out[0] = r0 + m;
        acc_out[1] = g0 + n;
    }
    const float *pr = step_rows(s, k);
    const uint8_t *t = tp + static_cast<int64_t>(k) * s.max_det * 10;
    for (int j = threadIdx.x; j < m; j += blockDim.x) {
        const long long at = r0 + j;
        if (at >= row_cap) break;
        conf[at] = pr[j * 6 + 4];
        pred_cls[at] = pr[j * 6 + 5];
    }
    for (int e = threadIdx.x; e < m * 10; e += blockDim.x) {
        const long long at = r0 * 10 + e;
        if (at >= row_cap * 10) break;
        tp_out[at] = t[e];
    }
    const T *g = static_cast<const T *>(s.d_gt) + static_cast<int64_t>(k) * s.max_gt * 5;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const long long at = g0 + i;
        if (at >= target_cap) break;
        target_cls[at] = static_cast<double>(g[static_cast<int64_t>(i) * 5 + 4]);
    }
}

cudaError_t launch_map_iou(const void *b1, int64_t n, int w1, const void *b2, int64_t m, int w2, int f64, void *out,
                           cudaStream_t stream)
{
    if (n == 0 || m == 0) return cudaSuccess;
    for (int64_t r0 = 0; r0 < n; r0 += 65535) {
        const int64_t rows = (n - r0) < 65535 ? (n - r0) : 65535;
        const dim3 grid(static_cast<unsigned>((m + 255) / 256), static_cast<unsigned>(rows));
        if (f64)
            k_map_iou<double><<<grid, 256, 0, stream>>>(static_cast<const double *>(b1) + r0 * w1, rows, w1,
                                                        static_cast<const double *>(b2), m, w2,
                                                        static_cast<double *>(out) + r0 * m);
        else
            k_map_iou<float><<<grid, 256, 0, stream>>>(static_cast<const float *>(b1) + r0 * w1, rows, w1,
                                                       static_cast<const float *>(b2), m, w2,
                                                       static_cast<float *>(out) + r0 * m);
    }
    return cudaGetLastError();
}

cudaError_t launch_compute_tp(const void *gt, const int64_t *gt_off, const void *pred, const int64_t *pred_off, int batch,
                              int f64, const double *thr10, int32_t *first_pred, uint8_t *tp, cudaStream_t stream)
{
    if (batch == 0) return cudaSuccess;
    TpThresholds t;
    for (int i = 0; i < 10; ++i) t.v[i] = thr10[i];
    if (f64)
        k_compute_tp<double><<<batch, 256, 0, stream>>>(static_cast<const double *>(gt), gt_off,
                                                        static_cast<const double *>(pred), pred_off, t, first_pred, tp);
    else
        k_compute_tp<float><<<batch, 256, 0, stream>>>(static_cast<const float *>(gt), gt_off,
                                                       static_cast<const float *>(pred), pred_off, t, first_pred, tp);
    return cudaGetLastError();
}

cudaError_t launch_match_tp(const ysb_match_step &s, const double *thr10, int32_t *first_pred, uint8_t *tp,
                            cudaStream_t stream)
{
    const int images = s.world * s.batch;
    if (images == 0) return cudaSuccess;
    TpThresholds t;
    for (int i = 0; i < 10; ++i) t.v[i] = thr10[i];
    if (s.gt_dtype == YSB_F64)
        k_match_tp<double><<<images, 256, 0, stream>>>(s, t, first_pred, tp);
    else
        k_match_tp<float><<<images, 256, 0, stream>>>(s, t, first_pred, tp);
    return cudaGetLastError();
}

cudaError_t launch_match_compact(const ysb_match_step &s, const uint8_t *tp, const int64_t *acc_in, int64_t *acc_out,
                                 float *conf, float *pred_cls, uint8_t *tp_out, int64_t row_cap, double *target_cls,
                                 int64_t target_cap, cudaStream_t stream)
{
    const int images = s.world * s.batch;
    if (images == 0) return cudaMemcpyAsync(acc_out, acc_in, 2 * sizeof(int64_t), cudaMemcpyDeviceToDevice, stream);
    const long long *ai = reinterpret_cast<const long long *>(acc_in);
    long long *ao = reinterpret_cast<long long *>(acc_out);
    if (s.gt_dtype == YSB_F64)
        k_match_compact<double><<<images, 256, 0, stream>>>(s, tp, ai, ao, conf, pred_cls, tp_out, row_cap, target_cls,
                                                            target_cap);
    else
        k_match_compact<float><<<images, 256, 0, stream>>>(s, tp, ai, ao, conf, pred_cls, tp_out, row_cap, target_cls,
                                                           target_cap);
    return cudaGetLastError();
}

// ---- weighted-box-fusion, utils/weighted_fusion_bbox.py:41-96 -----------------------------------------------------------
// Rows are (x1, y1, x2, y2, score, label, weight[, order]) float32; image i owns rows [i*stride, i*stride + counts[i]).
// The reference walks every label's boxes in descending score order; a box joins EVERY cluster whose current fused box
// it overlaps by IoU >= thr (cpu_iou, utils/bbox_tools.py:63-84: float32 area of the box, float64 everything else,
// union clipped at 1e-6), or founds a new cluster; after every box all fused boxes are recomputed
// (update_fusion_bbox :41-60: mean over members of box*score/sum(score) -- the score-weighted mean divided by the member
// count once more -- and sum(score*weight)/sum(weight)).  Here: (1) a rank sort orders every image by (label asc, score
// desc, later row first: argsort()[::-1] of a stable sort), (2) one warp per (image, label) segment walks it, lanes
// strided over the clusters, cluster sums kept incrementally in float64.
struct WbfCluster {
    double a[4];     // sum box * score
    double s;        // sum score
    double sw;       // sum score * weight
    double w;        // sum weight
    double fus[4];   // current fused box
    int cnt;
    int pad;
};

__device__ __forceinline__ uint32_t sortable_f32(float v)
{
    const uint32_t b = __float_as_uint(v);
    return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}

__global__ void __launch_bounds__(256) k_wbf_keys(const float *__restrict__ rows, int row_w, const int32_t *__restrict__ counts,
                                                  int64_t stride, uint64_t *__restrict__ k1, uint32_t *__restrict__ k2)
{
    const int img = blockIdx.y;
    const int64_t j = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (j >= counts[img]) return;
    const float *r = rows + (static_cast<int64_t>(img) * stride + j) * row_w;
    const int label = static_cast<int>(r[5]);
    k1[img * stride + j] = (static_cast<uint64_t>(static_cast<uint32_t>(0x7fffffff - label)) << 32) | sortable_f32(r[4]);
    k2[img * stride + j] = row_w >= 8 ? __float_as_uint(r[7]) : static_cast<uint32_t>(j);
}

// rank = number of rows of the image that sort before this one (descending (k1, k2)); keys are distinct per image.
__global__ void __launch_bounds__(256) k_wbf_rank(const int32_t *__restrict__ counts, int64_t stride,
                                                  const uint64_t *__restrict__ k1, const uint32_t *__restrict__ k2,
                                                  int32_t *__restrict__ order, uint64_t *__restrict__ sorted_k1)
{
    const int img = blockIdx.y;
    const int n = counts[img];
    const int64_t j = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (j >= n) return;
    const uint64_t *a1 = k1 + img * stride;
    const uint32_t *a2 = k2 + img * stride;
    const uint64_t m1 = a1[j];
    const uint32_t m2 = a2[j];
    int rank = 0;
    for (int i = 0; i < n; ++i) {
        const uint64_t o1 = __ldg(a1 + i);
        rank += (o1 > m1 || (o1 == m1 && __ldg(a2 + i) > m2)) ? 1 : 0;
    }
    order[img * stride + rank] = static_cast<int32_t>(j);
    sorted_k1[img * stride + rank] = m1;
}

// cpu_iou(box (float32), fused (float64)), utils/bbox_tools.py:63-84
__device__ __forceinline__ double wbf_iou(const float *b, const double *f)
{
    const double a1 = static_cast<double>(__fmul_rn(__fsub_rn(b[2], b[0]), __fsub_rn(b[3], b[1])));  // np.prod of float32 sides
    const double a2 = (f[2] - f[0]) * (f[3] - f[1]);
    const double bx1 = b[0], by1 = b[1], bx2 = b[2], by2 = b[3];
    const double ymax = by2 < f[3] ? by2 : f[3], xmax = bx2 < f[2] ? bx2 : f[2];
    const double ymin = by1 > f[1] ? by1 : f[1], xmin = bx1 > f[0] ? bx1 : f[0];
    double w = xmax - xmin, h = ymax - ymin;
    w = w > 0.0 ? w : 0.0;
    h = h > 0.0 ? h : 0.0;
    const double inter = w * h;
    double den = a1 + a2 - inter;
    den = den < 1e-6 ? 1e-6 : den;
    return inter / den;
}

// One warp per sorted position; only the warps that sit on the first row of a label segment work.
__global__ void __launch_bounds__(256) k_wbf_cluster(const float *__restrict__ rows, int row_w, const int32_t *__restrict__ counts,
                                                     int64_t stride, double thr, const int32_t *__restrict__ order,
                                                     const uint64_t *__restrict__ sorted_k1, WbfCluster *__restrict__ clusters,
                                                     double *__restrict__ fusion, int32_t *__restrict__ members,
                                                     int32_t *__restrict__ pairs, long long pair_cap,
                                                     unsigned long long *__restrict__ pair_count, int32_t *__restrict__ status)
{
    const int img = blockIdx.y;
    const int n = counts[img];
    const int64_t p0 = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (p0 >= n) return;
    const int64_t base = static_cast<int64_t>(img) * stride;
    const uint32_t lab_key = static_cast<uint32_t>(sorted_k1[base + p0] >> 32);
    if (p0 > 0 && static_cast<uint32_t>(sorted_k1[base + p0 - 1] >> 32) == lab_key) return;   // not a segment start
    int64_t p1 = p0 + 1;
    while (p1 < n && static_cast<uint32_t>(sorted_k1[base + p1] >> 32) == lab_key) ++p1;
    WbfCluster *cl = clusters + base + p0;
    // fusion_bbox = [top box], cluster_bbox = [[]] (:73-74)
    const float *top = rows + (base + order[base + p0]) * row_w;
    if (lane == 0) {
        WbfCluster c{};
        for (int q = 0; q < 4; ++q) c.fus[q] = static_cast<double>(top[q]);
        cl[0] = c;
    }
    __syncwarp();
    int nclus = 1;
    bool broken = false;
    for (int64_t k = p0; k < p1; ++k) {
        const float *r = rows + (base + order[base + k]) * row_w;
        const double sc = static_cast<double>(r[4]), wt = static_cast<double>(r[6]);
        bool hit_any = false;
        for (int c = lane; c < nclus; c += 32) {
            WbfCluster &C = cl[c];
            if (wbf_iou(r, C.fus) >= thr) {
                hit_any = true;
                for (int q = 0; q < 4; ++q) C.a[q] += static_cast<double>(r[q]) * sc;
                C.s += sc;
                C.sw += sc * wt;
                C.w += wt;
                C.cnt += 1;
                for (int q = 0; q < 4; ++q) C.fus[q] = C.a[q] / C.s / static_cast<double>(C.cnt);
                if (pairs) {
                    const unsigned long long at = atomicAdd(pair_count, 1ull);
                    if (at < static_cast<unsigned long long>(pair_cap)) {
                        pairs[2 * at] = static_cast<int32_t>(base + p0 + c);   // global slot / position indices
                        pairs[2 * at + 1] = static_cast<int32_t>(base + k);
                    }
                }
            }
        }
        hit_any = __any_sync(0xffffffffu, hit_any);
        if (!hit_any) {
            if (k == p0) { broken = true; break; }   // the top box misses itself: cluster 0 stays empty, the reference raises
            if (lane == 0) {
                WbfCluster c{};
                for (int q = 0; q < 4; ++q) { c.a[q] = static_cast<double>(r[q]) * sc; }
                c.s = sc;
                c.sw = sc * wt;
                c.w = wt;
                c.cnt = 1;
                for (int q = 0; q < 4; ++q) c.fus[q] = c.a[q] / c.s / 1.0;
                cl[nclus] = c;
                if (pairs) {
                    const unsigned long long at = atomicAdd(pair_count, 1ull);
                    if (at < static_cast<unsigned long long>(pair_cap)) {
                        pairs[2 * at] = static_cast<int32_t>(base + p0 + nclus);
                        pairs[2 * at + 1] = static_cast<int32_t>(base + k);
                    }
                }
            }
            ++nclus;
        }
        __syncwarp();
    }
    if (broken) {
        if (lane == 0) atomicExch(status + img, 1);
        return;
    }
    const double label = static_cast<double>(top[5]);
    for (int c = lane; c < nclus; c += 32) {
        const WbfCluster &C = cl[c];
        double *f = fusion + (base + p0 + c) * 6;
        for (int q = 0; q < 4; ++q) f[q] = C.fus[q];
        f[4] = C.sw / C.w;
        f[5] = label;
        members[base + p0 + c] = C.cnt;
    }
}

// do_wfb's per-pass filter (trainer/eval_yolov5.py:57-79; v7 / YOLOX identical) on the decoded rows of all passes:
// obj > thr, conf = cls * obj (float32), best class (first maximum) with conf > thr -- or, mutil_label, every class above
// it --, xywh -> xyxy, the pass weight; one record per survivor appended to the image's list (order restored by the sort
// through column 7 = position in the reference's stacked list).
struct WbfPasses {
    long long first_row[YSB_MAX_PASSES + 1];
    float weight[YSB_MAX_PASSES];
    int n;
};

__global__ void __launch_bounds__(256) k_wbf_collect(const float *__restrict__ decoded, int64_t rows, int row_w, int C,
                                                     float thr, int multi, const __grid_constant__ WbfPasses passes,
                                                     float *__restrict__ rec, int32_t *__restrict__ counts, int64_t cap)
{
    const int img = blockIdx.y;
    const int64_t j = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (j >= rows) return;
    const float *r = decoded + (static_cast<int64_t>(img) * rows + j) * row_w;
    const float obj = r[4];
    if (!(obj > thr)) return;
    float weight = passes.weight[0];
    for (int q = 1; q < passes.n; ++q)
        if (j >= passes.first_row[q]) weight = passes.weight[q];
    const float hw = __fmul_rn(r[2], 0.5f), hh = __fmul_rn(r[3], 0.5f);   // w / 2 is exact either way
    const float x1 = __fsub_rn(r[0], hw), y1 = __fsub_rn(r[1], hh), x2 = __fadd_rn(r[0], hw), y2 = __fadd_rn(r[1], hh);
    auto emit = [&](float conf, int cls, uint32_t pos) {
        const int at = atomicAdd(counts + img, 1);
        if (at >= cap) return;
        float *o = rec + (static_cast<int64_t>(img) * cap + at) * 8;
        o[0] = x1; o[1] = y1; o[2] = x2; o[3] = y2;
        o[4] = conf;
        o[5] = static_cast<float>(cls);
        o[6] = weight;
        o[7] = __uint_as_float(pos);
    };
    if (multi) {
        for (int k = 0; k < C; ++k) {
            const float conf = __fmul_rn(r[5 + k], obj);
            if (conf > thr) emit(conf, k, static_cast<uint32_t>(j) * static_cast<uint32_t>(C) + static_cast<uint32_t>(k));
        }
    } else {
        float best = __fmul_rn(r[5], obj);
        int bk = 0;
        for (int k = 1; k < C; ++k) {
            const float conf = __fmul_rn(r[5 + k], obj);
            if (conf > best) { best = conf; bk = k; }
        }
        if (best > thr) emit(best, bk, static_cast<uint32_t>(j));
    }
}

size_t wbf_workspace_bytes(int batch, int64_t stride)
{
    const size_t slots = static_cast<size_t>(batch) * static_cast<size_t>(stride);
    return slots * (sizeof(WbfCluster) + 2 * sizeof(uint64_t) + sizeof(uint32_t)) + 64;
}

cudaError_t launch_wbf(const float *rows, int row_w, const int32_t *counts, int batch, int64_t stride, double thr, void *ws,
                       int32_t *order, double *fusion, int32_t *members, int32_t *pairs, long long pair_cap,
                       unsigned long long *pair_count, int32_t *status, cudaStream_t stream)
{
    if (batch == 0 || stride == 0) return cudaSuccess;
    const size_t slots = static_cast<size_t>(batch) * static_cast<size_t>(stride);
    WbfCluster *clusters = static_cast<WbfCluster *>(ws);
    uint64_t *k1 = reinterpret_cast<uint64_t *>(clusters + slots);
    uint64_t *sk1 = k1 + slots;
    uint32_t *k2 = reinterpret_cast<uint32_t *>(sk1 + slots);
    cudaError_t e = cudaMemsetAsync(status, 0, sizeof(int32_t) * batch, stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(members, 0, sizeof(int32_t) * slots, stream);
    if (e == cudaSuccess && pair_count) e = cudaMemsetAsync(pair_count, 0, sizeof(unsigned long long), stream);
    if (e != cudaSuccess) return e;
    const dim3 g1(static_cast<unsigned>((stride + 255) / 256), static_cast<unsigned>(batch));
    k_wbf_keys<<<g1, 256, 0, stream>>>(rows, row_w, counts, stride, k1, k2);
    k_wbf_rank<<<g1, 256, 0, stream>>>(counts, stride, k1, k2, order, sk1);
    const dim3 g2(static_cast<unsigned>((stride * 32 + 255) / 256), static_cast<unsigned>(batch));
    k_wbf_cluster<<<g2, 256, 0, stream>>>(rows, row_w, counts, stride, thr, order, sk1, clusters, fusion, members, pairs,
                                          pair_cap, pair_count, status);
    return cudaGetLastError();
}

cudaError_t launch_wbf_collect(const float *decoded, int batch, int64_t rows, int row_w, int C, float thr, int multi,
                               const int64_t *pass_rows, const float *pass_weights, int n_pass, float *rec, int32_t *counts,
                               int64_t cap, cudaStream_t stream)
{
    cudaError_t e = cudaMemsetAsync(counts, 0, sizeof(int32_t) * (batch > 0 ? batch : 1), stream);
    if (e != cudaSuccess || batch == 0 || rows == 0) return e;
    WbfPasses P{};
    P.n = n_pass;
    long long at = 0;
    for (int q = 0; q < n_pass; ++q) {
        P.first_row[q] = at;
        P.weight[q] = pass_weights[q];
        at += pass_rows[q];
    }
    P.first_row[n_pass] = at;
    const dim3 grid(static_cast<unsigned>((rows + 255) / 256), static_cast<unsigned>(batch));
    k_wbf_collect<<<grid, 256, 0, stream>>>(decoded, rows, row_w, C, thr, multi, P, rec, counts, cap);
    return cudaGetLastError();
}

}  // namespace ysb
