// gather_kernels.cu -- the one exchange of the multi-GPU path: all-gather of the kept detections, without a collective
// launch (SURVEY.md 8e; include/ysb_postproc.h "multi-GPU").
//
// Every rank owns one symmetric receive buffer, mapped by its peers through CUDA IPC (NVLink P2P).  The producer side
// lives in the NMS kernel (nms_kernel.cu: the ordered row write stores into every peer's slot and then adds one
// system-scope arrival count per image); this file holds the buffer management and the flow-control kernels:
//   k_gather_begin  zero the filter counters of the step; publish "I am done reading the previous use of this slot"
//                   (ack) to every peer.  The NMS kernel waits for the peers' acks before it overwrites their slots.
//   k_gather_wait   wait until all images of every rank have landed in my slot; bump the slot's use counter
//   k_gather_absent (partial steps) mark this rank's images beyond the ones it had as absent in every slot, and count
//                   them as arrived
// Spins are volatile loads of LOCAL memory that peers write remotely (the L2 is the point of coherence for incoming
// NVLink writes), bounded by a wall-clock limit: a timeout sets the buffer's err word instead of hanging the GPU.
#include <cstring>

#include "ysb_internal.cuh"

namespace ysb {

struct BeginArgs {
    int world, rank;
    unsigned int *peer_ack[YSB_MAX_PEERS];   // peer r's ack word for (slot, this rank)
    const unsigned int *my_ack;              // my ack words of this slot: [world]
    const unsigned int *use;                 // completed uses of this slot (local)
    unsigned int *err;
    int32_t *counts;
    long long n_counts;
};

__global__ void __launch_bounds__(256) k_gather_begin(const __grid_constant__ BeginArgs a)
{
    for (long long i = threadIdx.x; i < a.n_counts; i += blockDim.x) a.counts[i] = 0;
    const unsigned int u = *a.use;   // uses of this slot that I have completely consumed (stream order)
    const int r = threadIdx.x;
    // remote store: "rank `rank` is done with use u of this slot".  Nobody waits here: the matching wait sits in the NMS
    // kernel, right before its first store into a peer's slot (nms_kernel.cu), a whole filter + NMS pass later -- by then
    // the peers' acks have long arrived and the step-start barrier this used to be costs nothing.
    if (r < a.world && r != a.rank) *reinterpret_cast<volatile unsigned int *>(a.peer_ack[r]) = u;
}

struct WaitArgs {
    int world, batch;
    const unsigned int *arrived;   // my arrival counters of this slot: [world]
    unsigned int *use;
    unsigned int *err;
};

__global__ void __launch_bounds__(32) k_gather_wait(const __grid_constant__ WaitArgs a)
{
    const unsigned int u = *a.use;
    const unsigned int target = (u + 1u) * static_cast<unsigned int>(a.batch);
    const int r = threadIdx.x;
    if (r < a.world && !spin_until_reached(a.arrived + r, target)) atomicExch(a.err, 2u);
    __threadfence_system();   // the rows behind the counters are visible to everything that follows on this stream
    __syncwarp();
    if (r == 0) *a.use = u + 1u;
}

// Images [first, batch) of this rank are absent from this step (a partial step, ysb_select_nms_gather_partial): the
// M <= 0 branch of k_select_nms for a range of images, with the absent mark instead of -1.  Once per peer: wait for its
// ack of this slot, then YSB_CNT_ABSENT into every rank's count words of those images, then one arrival increment of
// batch - first, so k_gather_wait's target (use + 1) * batch and the ack protocol of later steps hold unchanged.
__global__ void __launch_bounds__(256) k_gather_absent(const __grid_constant__ GatherSink G, int first, int batch)
{
    const int tid = threadIdx.x;
    if (tid < G.world && tid != G.rank && !spin_until_reached(G.my_ack + tid, *G.use)) atomicExch(G.err, 1u);
    __syncthreads();
    const int n = batch - first;
    for (int e = tid; e < G.world * n; e += blockDim.x) G.cnt[e / n][first + e % n] = YSB_CNT_ABSENT;
    __threadfence_system();   // release: the marks are ordered before the arrival counts the peers wait for
    __syncthreads();
    if (tid < G.world) atomicAdd_system(G.arrived[tid], static_cast<unsigned int>(n));
}

static bool gather_ok(const ysb_gather *g, int slot)
{
    if (!g || g->world < 1 || g->world > YSB_MAX_PEERS || g->rank < 0 || g->rank >= g->world) return false;
    if (g->slots < 1 || slot < 0 || slot >= g->slots || g->batch < 0 || g->max_det <= 0) return false;
    for (int r = 0; r < g->world; ++r)
        if (!g->d_buf[r]) return false;
    return true;
}

static inline unsigned char *at(void *base, size_t off) { return static_cast<unsigned char *>(base) + off; }

bool make_gather_sink(const ysb_gather *g, int slot, GatherSink *out)
{
    if (!gather_ok(g, slot)) return false;
    const GatherLayout L = gather_layout(g->world, g->slots, g->batch, g->max_det);
    std::memset(out, 0, sizeof(*out));
    out->world = g->world;
    out->rank = g->rank;
    for (int r = 0; r < g->world; ++r) {
        out->rows[r] = reinterpret_cast<float *>(at(g->d_buf[r], L.rows + L.rows_slot * slot + L.rows_rank * g->rank));
        out->cnt[r] = reinterpret_cast<int32_t *>(at(g->d_buf[r], L.cnt + L.cnt_slot * slot + L.cnt_rank * g->rank));
        out->arrived[r] = reinterpret_cast<unsigned int *>(at(g->d_buf[r], L.arrived)) + (static_cast<size_t>(slot) * g->world + g->rank);
    }
    void *mine = g->d_buf[g->rank];
    out->my_ack = reinterpret_cast<unsigned int *>(at(mine, L.ack)) + static_cast<size_t>(slot) * g->world;
    out->use = reinterpret_cast<unsigned int *>(at(mine, L.use)) + slot;
    out->err = reinterpret_cast<unsigned int *>(at(mine, L.err));
    return true;
}

cudaError_t launch_gather_begin(const ysb_gather *g, int slot, int32_t *d_counts, int64_t n_counts, cudaStream_t stream)
{
    const GatherLayout L = gather_layout(g->world, g->slots, g->batch, g->max_det);
    BeginArgs a;
    std::memset(&a, 0, sizeof(a));
    a.world = g->world;
    a.rank = g->rank;
    void *mine = g->d_buf[g->rank];
    for (int r = 0; r < g->world; ++r)
        a.peer_ack[r] = reinterpret_cast<unsigned int *>(at(g->d_buf[r], L.ack)) + (static_cast<size_t>(slot) * g->world + g->rank);
    a.my_ack = reinterpret_cast<unsigned int *>(at(mine, L.ack)) + static_cast<size_t>(slot) * g->world;
    a.use = reinterpret_cast<unsigned int *>(at(mine, L.use)) + slot;
    a.err = reinterpret_cast<unsigned int *>(at(mine, L.err));
    a.counts = d_counts;
    a.n_counts = d_counts ? n_counts : 0;
    k_gather_begin<<<1, 256, 0, stream>>>(a);
    return cudaGetLastError();
}

cudaError_t launch_gather_wait(const ysb_gather *g, int slot, cudaStream_t stream)
{
    const GatherLayout L = gather_layout(g->world, g->slots, g->batch, g->max_det);
    WaitArgs a;
    void *mine = g->d_buf[g->rank];
    a.world = g->world;
    a.batch = g->batch;
    a.arrived = reinterpret_cast<unsigned int *>(at(mine, L.arrived)) + static_cast<size_t>(slot) * g->world;
    a.use = reinterpret_cast<unsigned int *>(at(mine, L.use)) + slot;
    a.err = reinterpret_cast<unsigned int *>(at(mine, L.err));
    k_gather_wait<<<1, 32, 0, stream>>>(a);
    return cudaGetLastError();
}

cudaError_t launch_gather_absent(const GatherSink &sink, int first, int batch, cudaStream_t stream)
{
    if (first >= batch) return cudaSuccess;
    k_gather_absent<<<1, 256, 0, stream>>>(sink, first, batch);
    return cudaGetLastError();
}

bool gather_valid(const ysb_gather *g, int slot) { return gather_ok(g, slot); }

}  // namespace ysb
