// comm.cu -- the multi-GPU exchange step of the path in the C ABI (rtb_comm_* in include/rtb.h, SURVEY.md 8(b)(iv), 8(e)).
//
// Rays shard by contiguous index range over one process per GPU and the trace itself never communicates; what is
// exchanged afterwards are the reduced products only: the (3, G, G) pupil grid (a sum) and the 12-entry statistics vectors
// (8 sums, 2 minima, 2 maxima).  The grid is one ncclAllReduce(sum, double) in place; the statistics of every bucket are
// one ncclAllGather into scratch followed by a merge kernel -- two collectives per step instead of four.
//
// NCCL is resolved at run time (dlopen "libnccl.so.2"): a process that has PyTorch loaded shares the copy PyTorch
// brought, any other binder gets the system library, and librtb.so itself loads on machines without NCCL (every rtb_comm_*
// call then fails with RTB_ERR_UNSUPPORTED).  Bootstrapping is the caller's: rank 0 asks rtb_comm_unique_id for 128
// bytes and hands them to the other ranks by whatever it has (MPI, a file, torch.distributed's store).
#include <dlfcn.h>

#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <mutex>

#include <math_constants.h>
#include <nccl.h>

#include "rtb_device.cuh"

namespace {

struct NcclApi {
    void *handle = nullptr;
    ncclResult_t (*GetVersion)(int *) = nullptr;
    ncclResult_t (*GetUniqueId)(ncclUniqueId *) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t *, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*CommCount)(const ncclComm_t, int *) = nullptr;
    ncclResult_t (*AllReduce)(const void *, void *, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*AllGather)(const void *, void *, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
    const char *(*GetErrorString)(ncclResult_t) = nullptr;
    bool ok = false;
};

NcclApi g_nccl;
std::once_flag g_nccl_once;

const NcclApi &nccl()
{
    std::call_once(g_nccl_once, [] {
        NcclApi &n = g_nccl;
        for (const char *name : {"libnccl.so.2", "libnccl.so"}) {
            n.handle = dlopen(name, RTLD_NOW | RTLD_GLOBAL);
            if (n.handle) break;
        }
        if (!n.handle) return;
        auto sym = [&](const char *s) { return dlsym(n.handle, s); };
        n.GetVersion = (decltype(n.GetVersion))sym("ncclGetVersion");
        n.GetUniqueId = (decltype(n.GetUniqueId))sym("ncclGetUniqueId");
        n.CommInitRank = (decltype(n.CommInitRank))sym("ncclCommInitRank");
        n.CommDestroy = (decltype(n.CommDestroy))sym("ncclCommDestroy");
        n.CommCount = (decltype(n.CommCount))sym("ncclCommCount");
        n.AllReduce = (decltype(n.AllReduce))sym("ncclAllReduce");
        n.AllGather = (decltype(n.AllGather))sym("ncclAllGather");
        n.GetErrorString = (decltype(n.GetErrorString))sym("ncclGetErrorString");
        n.ok = n.GetVersion && n.GetUniqueId && n.CommInitRank && n.CommDestroy && n.CommCount && n.AllReduce &&
               n.AllGather && n.GetErrorString;
    });
    return g_nccl;
}

// gathered: [rank][bucket][12] -> stats[bucket][12]: entries 0-7 summed in rank order (deterministic), 8 / 10 minima,
// 9 / 11 maxima (include/rtb.h: rtb_reduce)
__global__ void merge_stats_kernel(const double *gathered, double *stats, int n_ranks, int n_buckets)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_buckets * RTB_N_STATS) return;
    const int k = i % RTB_N_STATS;
    double acc = gathered[i];
    for (int r = 1; r < n_ranks; r++) {
        const double v = gathered[(size_t)r * n_buckets * RTB_N_STATS + i];
        acc = (k < 8) ? acc + v : ((k == 8 || k == 10) ? fmin(acc, v) : fmax(acc, v));
    }
    stats[i] = acc;
}

} // namespace

struct rtb_comm {
    ncclComm_t comm = nullptr;
    int n_ranks = 0, rank = 0, device = 0;
    double *scratch = nullptr;      // all-gather landing zone for the statistics
    size_t scratch_doubles = 0;
};

#define RTB_NCCL(call)                                                                                            \
    do {                                                                                                          \
        ncclResult_t r_ = (call);                                                                                 \
        if (r_ != ncclSuccess)                                                                                    \
            return rtb::api_fail(RTB_ERR_CUDA, "%s failed: %s", #call, nccl().GetErrorString(r_));                \
    } while (0)

extern "C" {

int rtb_comm_available(void)
{
    const NcclApi &n = nccl();
    if (!n.ok) return 0;
    int v = 0;
    return n.GetVersion(&v) == ncclSuccess ? v : 0;
}

int rtb_comm_unique_id(void *id_out, size_t id_bytes)
{
    if (!id_out || id_bytes < RTB_COMM_ID_BYTES) return rtb::api_fail(RTB_ERR_INVALID, "id_out needs %d bytes", RTB_COMM_ID_BYTES);
    const NcclApi &n = nccl();
    if (!n.ok) return rtb::api_fail(RTB_ERR_UNSUPPORTED, "NCCL (libnccl.so.2) is not available in this process");
    static_assert(RTB_COMM_ID_BYTES == NCCL_UNIQUE_ID_BYTES, "rtb.h and nccl.h disagree on the id size");
    ncclUniqueId id;
    RTB_NCCL(n.GetUniqueId(&id));
    memcpy(id_out, &id, sizeof(id));
    return RTB_OK;
}

int rtb_comm_init(rtb_comm **comm_out, int n_ranks, int rank, const void *unique_id, int device)
{
    if (!comm_out || !unique_id) return rtb::api_fail(RTB_ERR_INVALID, "NULL argument");
    if (n_ranks < 1 || rank < 0 || rank >= n_ranks) return rtb::api_fail(RTB_ERR_INVALID, "rank %d of %d", rank, n_ranks);
    const NcclApi &n = nccl();
    if (!n.ok) return rtb::api_fail(RTB_ERR_UNSUPPORTED, "NCCL (libnccl.so.2) is not available in this process");
    int n_dev = 0;
    if (cudaGetDeviceCount(&n_dev) != cudaSuccess || device < 0 || device >= n_dev)
        return rtb::api_fail(RTB_ERR_INVALID, "device index %d (of %d visible)", device, n_dev);
    int prev = 0;
    cudaGetDevice(&prev);
    cudaSetDevice(device);
    ncclUniqueId id;
    memcpy(&id, unique_id, sizeof(id));
    rtb_comm *c = new rtb_comm;
    ncclResult_t r = n.CommInitRank(&c->comm, n_ranks, id, rank);
    cudaSetDevice(prev);
    if (r != ncclSuccess) {
        delete c;
        return rtb::api_fail(RTB_ERR_CUDA, "ncclCommInitRank failed: %s", n.GetErrorString(r));
    }
    c->n_ranks = n_ranks;
    c->rank = rank;
    c->device = device;
    *comm_out = c;
    return RTB_OK;
}

int rtb_comm_size(const rtb_comm *comm)
{
    if (!comm) return rtb::api_fail(RTB_ERR_INVALID, "comm is NULL");
    int count = 0;
    RTB_NCCL(nccl().CommCount(comm->comm, &count));
    return count;
}

int rtb_comm_allreduce_grid(rtb_comm *comm, double *grid_dev, int64_t n_doubles, void *stream)
{
    if (!comm || (!grid_dev && n_doubles > 0) || n_doubles < 0) return rtb::api_fail(RTB_ERR_INVALID, "bad arguments");
    if (n_doubles == 0 || comm->n_ranks == 1) return RTB_OK;
    RTB_NCCL(nccl().AllReduce(grid_dev, grid_dev, (size_t)n_doubles, ncclDouble, ncclSum, comm->comm, (cudaStream_t)stream));
    return RTB_OK;
}

int rtb_comm_allreduce_stats(rtb_comm *comm, double *stats_dev, int n_buckets, void *stream)
{
    if (!comm || !stats_dev || n_buckets < 1) return rtb::api_fail(RTB_ERR_INVALID, "bad arguments");
    if (comm->n_ranks == 1) return RTB_OK;
    const size_t per_rank = (size_t)n_buckets * RTB_N_STATS;
    const size_t need = per_rank * (size_t)comm->n_ranks;
    int prev = 0;
    cudaGetDevice(&prev);
    cudaSetDevice(comm->device);
    if (comm->scratch_doubles < need) {
        // (grows only; a buffer still in use by an earlier call on another stream would have to be synchronised first)
        if (comm->scratch) {
            cudaDeviceSynchronize();
            cudaFree(comm->scratch);
        }
        comm->scratch = nullptr;
        comm->scratch_doubles = 0;
        if (cudaMalloc((void **)&comm->scratch, need * sizeof(double)) != cudaSuccess) {
            cudaSetDevice(prev);
            return rtb::api_fail(RTB_ERR_NOMEM, "cudaMalloc of %zu bytes failed", need * sizeof(double));
        }
        comm->scratch_doubles = need;
    }
    ncclResult_t r = nccl().AllGather(stats_dev, comm->scratch, per_rank, ncclDouble, comm->comm, (cudaStream_t)stream);
    cudaError_t e = cudaSuccess;
    if (r == ncclSuccess) {
        const int threads = 128, blocks = (int)((per_rank + threads - 1) / threads);
        merge_stats_kernel<<<blocks, threads, 0, (cudaStream_t)stream>>>(comm->scratch, stats_dev, comm->n_ranks, n_buckets);
        e = cudaGetLastError();
    }
    cudaSetDevice(prev);
    if (r != ncclSuccess) return rtb::api_fail(RTB_ERR_CUDA, "ncclAllGather failed: %s", nccl().GetErrorString(r));
    if (e != cudaSuccess) return rtb::api_fail(RTB_ERR_CUDA, "statistics merge launch failed: %s", cudaGetErrorString(e));
    return RTB_OK;
}

int rtb_comm_destroy(rtb_comm *comm)
{
    if (!comm) return RTB_OK;
    if (comm->scratch) cudaFree(comm->scratch);
    ncclResult_t r = nccl().CommDestroy(comm->comm);
    delete comm;
    if (r != ncclSuccess) return rtb::api_fail(RTB_ERR_CUDA, "ncclCommDestroy failed: %s", nccl().GetErrorString(r));
    return RTB_OK;
}

} // extern "C"
