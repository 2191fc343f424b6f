// Multi-GPU exchange steps of the path, inside the library: one mesh partition per GPU (one process per GPU),
// NCCL over NVLink 5 / NVSwitch.
//
// What the reference gets from PETSc/MPI under `mpirun -n N` (SURVEY.md §2.4) and where it is triggered:
//   * forward ghost update of a block vector, owner -> ghost copies: `x.ghostUpdate(INSERT, FORWARD)`
//     (src/solvers/stabilized_schur.py:137-142,168)                      -> hemo_comm_halo_update
//   * sums of the Krylov / Newton reductions (VecMDot, VecNorm, VecDot inside KSPSolve / SNESSolve, :321)
//                                                                         -> hemo_comm_allreduce, hemo_global_dot
//   * assemble_scalar + comm.allreduce of the outlet flux (stabilized_schur_pressure_backflow.py:205,385)
//                                                                         -> hemo_comm_allreduce
// Local numbering of a partition: owned nodes first, then ghost nodes grouped by owner rank, so every receive lands
// directly in its slice of the vector (no unpack kernel); the send side packs boundary nodes with one gather kernel.
// Every NCCL call is enqueued on the context's stream and can be captured in the FGMRES iteration graph.
//
// NCCL is loaded with dlopen at hemo_comm_init (the process already holds torch's libnccl.so.2), so the
// single-GPU library has no link-time dependency on it.
#include <dlfcn.h>
#include <string.h>

#include "hemo_internal.cuh"

typedef struct ncclComm* ncclComm_t;
typedef struct { char internal[128]; } ncclUniqueId;
typedef int ncclResult_t;
enum { ncclFloat64 = 8, ncclSum = 0 };

struct NcclApi {
    void* lib = nullptr;
    ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*AllReduce)(const void*, void*, size_t, int, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*Send)(const void*, size_t, int, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*Recv)(void*, size_t, int, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*GroupStart)() = nullptr;
    ncclResult_t (*GroupEnd)() = nullptr;
    const char* (*GetErrorString)(ncclResult_t) = nullptr;
    ncclResult_t (*GetVersion)(int*) = nullptr;
};

static NcclApi g_nccl;

static const char* nccl_load() {
    if (g_nccl.lib) return nullptr;
    const char* names[] = {"libnccl.so.2", "libnccl.so"};
    void* h = nullptr;
    for (const char* nm : names) {
        h = dlopen(nm, RTLD_NOW | RTLD_GLOBAL | RTLD_NOLOAD);      // torch's copy, if the process has it
        if (!h) h = dlopen(nm, RTLD_NOW | RTLD_GLOBAL);
        if (h) break;
    }
    if (!h) return "libnccl.so.2 not found (import torch.distributed with the nccl backend first, or add NCCL to LD_LIBRARY_PATH)";
#define SYM(field, name)                                             \
    g_nccl.field = (decltype(g_nccl.field))dlsym(h, name);          \
    if (!g_nccl.field) return "NCCL symbol missing: " name;
    SYM(GetUniqueId, "ncclGetUniqueId")
    SYM(CommInitRank, "ncclCommInitRank")
    SYM(CommDestroy, "ncclCommDestroy")
    SYM(AllReduce, "ncclAllReduce")
    SYM(Send, "ncclSend")
    SYM(Recv, "ncclRecv")
    SYM(GroupStart, "ncclGroupStart")
    SYM(GroupEnd, "ncclGroupEnd")
    SYM(GetErrorString, "ncclGetErrorString")
    SYM(GetVersion, "ncclGetVersion")
#undef SYM
    g_nccl.lib = h;
    return nullptr;
}

#define HEMO_MAX_NEIGH 16

struct HemoComm {
    ncclComm_t comm = nullptr;
    int rank = 0, nranks = 1;
    // partition
    int n_owned = 0;
    int nneigh = 0;
    int peer[HEMO_MAX_NEIGH];
    int send_ptr[HEMO_MAX_NEIGH + 1];     // into send_nodes
    int recv_ptr[HEMO_MAX_NEIGH + 1];     // ghost node offsets (relative to n_owned)
    int32_t* send_nodes = nullptr;        // device, local node ids (owned)
    double* sendbuf = nullptr;            // device, (dim + 1) * total_send
    int64_t halo_updates = 0, allreduces = 0;
};

#define HEMO_CHECK_NCCL(ctx, expr)                                                     \
    do {                                                                               \
        ncclResult_t _r = (expr);                                                      \
        if (_r != 0) {                                                                 \
            (ctx)->err = std::string(#expr) + ": " + g_nccl.GetErrorString(_r);        \
            return 1000 + (int)_r;                                                     \
        }                                                                              \
    } while (0)

extern "C" int hemo_comm_unique_id(char* out128) {
    if (!out128) return HEMO_EINVAL;
    if (nccl_load()) return HEMO_ESTATE;
    ncclUniqueId id;
    if (g_nccl.GetUniqueId(&id) != 0) return HEMO_ESTATE;
    memcpy(out128, id.internal, 128);
    return 0;
}

extern "C" int hemo_comm_init(hemo_ctx* ctx, const char* uid128, int rank, int nranks) {
    if (!ctx || !uid128 || nranks < 1 || rank < 0 || rank >= nranks) return HEMO_EINVAL;
    const char* e = nccl_load();
    if (e) HEMO_FAIL(ctx, HEMO_ESTATE, e);
    hemo_comm_free(ctx);
    HemoComm* c = new HemoComm();
    c->rank = rank; c->nranks = nranks;
    ncclUniqueId id;
    memcpy(id.internal, uid128, 128);
    HEMO_CHECK_CUDA(ctx, cudaSetDevice(ctx->device));
    ncclResult_t r = g_nccl.CommInitRank(&c->comm, nranks, id, rank);
    if (r != 0) {
        ctx->err = std::string("ncclCommInitRank: ") + g_nccl.GetErrorString(r);
        delete c;
        return 1000 + (int)r;
    }
    ctx->comm = c;
    // the partitioned solve keeps plain launches: its chains interleave NCCL collectives with the library's kernels
    ctx->pdl = 0;
    return 0;
}

extern "C" int hemo_comm_info(hemo_ctx* ctx, int* rank, int* nranks, int* nccl_version, int64_t* halo_updates,
                              int64_t* allreduces) {
    if (!ctx || !ctx->comm) return HEMO_ESTATE;
    if (rank) *rank = ctx->comm->rank;
    if (nranks) *nranks = ctx->comm->nranks;
    if (nccl_version) g_nccl.GetVersion(nccl_version);
    if (halo_updates) *halo_updates = ctx->comm->halo_updates;
    if (allreduces) *allreduces = ctx->comm->allreduces;
    return 0;
}

void hemo_comm_free(hemo_ctx* ctx) {
    HemoComm* c = ctx->comm;
    if (!c) return;
    cudaStreamSynchronize(ctx->stream);
    cudaFree(c->send_nodes); cudaFree(c->sendbuf);
    if (c->comm && g_nccl.CommDestroy) g_nccl.CommDestroy(c->comm);
    delete c;
    ctx->comm = nullptr;
}

extern "C" int hemo_comm_set_partition(hemo_ctx* ctx, int n_owned, int nneigh, const int32_t* peers_host,
                                       const int32_t* send_ptr_host, const int32_t* send_nodes_host,
                                       const int32_t* recv_ptr_host, int ras_overlap) {
    if (!ctx || n_owned < 0 || nneigh < 0 || nneigh > HEMO_MAX_NEIGH) return HEMO_EINVAL;
    if (!ctx->comm) HEMO_FAIL(ctx, HEMO_ESTATE, "hemo_comm_init must precede hemo_comm_set_partition");
    if (!ctx->cells) HEMO_FAIL(ctx, HEMO_ESTATE, "hemo_set_mesh must precede hemo_comm_set_partition");
    if (n_owned > ctx->n) return HEMO_EINVAL;
    if (nneigh && (!peers_host || !send_ptr_host || !send_nodes_host || !recv_ptr_host)) return HEMO_EINVAL;
    HemoComm* c = ctx->comm;
    c->n_owned = n_owned;
    c->nneigh = nneigh;
    c->send_ptr[0] = c->recv_ptr[0] = 0;
    for (int k = 0; k < nneigh; ++k) {
        c->peer[k] = peers_host[k];
        c->send_ptr[k + 1] = send_ptr_host[k + 1];
        c->recv_ptr[k + 1] = recv_ptr_host[k + 1];
        if (c->peer[k] < 0 || c->peer[k] >= c->nranks || c->peer[k] == c->rank) return HEMO_EINVAL;
    }
    if (nneigh && n_owned + c->recv_ptr[nneigh] != ctx->n)
        HEMO_FAIL(ctx, HEMO_EINVAL, "ghost ranges do not cover the local nodes after the owned ones");
    const int total = nneigh ? c->send_ptr[nneigh] : 0;
    int rc;
    if ((rc = hemo_upload(ctx, &c->send_nodes, send_nodes_host, (size_t)total, false))) return rc;
    if ((rc = hemo_alloc(ctx, &c->sendbuf, (size_t)(ctx->dim + 1) * (total > 0 ? total : 1)))) return rc;
    HEMO_CHECK_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    // reductions run over the owned entries of [u (dim n) | p (n)]
    ctx->kry.seg_len0 = (int64_t)ctx->dim * n_owned;
    ctx->kry.seg_off1 = (int64_t)ctx->dim * ctx->n;
    ctx->kry.seg_len1 = n_owned;
    ctx->comm_ras_overlap = ras_overlap != 0;
    hemo_krylov_invalidate(ctx);
    return 0;
}

// sendbuf = [for each neighbour: u of its send nodes (dim each) | p of its send nodes]
__global__ void k_halo_pack(int total, int dim, int64_t n, const int32_t* __restrict__ nodes, const int* __restrict__ uoff,
                            const double* __restrict__ v, double* __restrict__ buf) {
    (void)uoff;
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= total) return;
    const int i = nodes[s];
    for (int k = 0; k < dim; ++k) buf[(int64_t)dim * s + k] = v[(int64_t)dim * i + k];
    buf[(int64_t)dim * total + s] = v[(int64_t)dim * n + i];
}

int hemo_comm_halo(hemo_ctx* ctx, double* v) {
    HemoComm* c = ctx->comm;
    if (!c) return 0;
    if (c->nneigh == 0) return 0;
    const int dim = ctx->dim;
    const int64_t n = ctx->n;
    const int total = c->send_ptr[c->nneigh];
    cudaStream_t st = ctx->stream;
    HEMO_PROF_BEGIN(ctx, HEMO_PROF_HALO);
    if (total > 0) {
        k_halo_pack<<<hemo_grid(total, 256), 256, 0, st>>>(total, dim, n, c->send_nodes, nullptr, v, c->sendbuf);
        HEMO_LAUNCH_CHECK(ctx);
    }
    HEMO_CHECK_NCCL(ctx, g_nccl.GroupStart());
    for (int k = 0; k < c->nneigh; ++k) {
        const int s0 = c->send_ptr[k], sc = c->send_ptr[k + 1] - s0;
        const int g0 = c->n_owned + c->recv_ptr[k], gc = c->recv_ptr[k + 1] - c->recv_ptr[k];
        if (sc > 0) {
            HEMO_CHECK_NCCL(ctx, g_nccl.Send(c->sendbuf + (int64_t)dim * s0, (size_t)dim * sc, ncclFloat64, c->peer[k], c->comm, st));
            HEMO_CHECK_NCCL(ctx, g_nccl.Send(c->sendbuf + (int64_t)dim * total + s0, (size_t)sc, ncclFloat64, c->peer[k], c->comm, st));
        }
        if (gc > 0) {
            HEMO_CHECK_NCCL(ctx, g_nccl.Recv(v + (int64_t)dim * g0, (size_t)dim * gc, ncclFloat64, c->peer[k], c->comm, st));
            HEMO_CHECK_NCCL(ctx, g_nccl.Recv(v + (int64_t)dim * n + g0, (size_t)gc, ncclFloat64, c->peer[k], c->comm, st));
        }
    }
    HEMO_CHECK_NCCL(ctx, g_nccl.GroupEnd());
    HEMO_PROF_END(ctx, HEMO_PROF_HALO);
    if (!ctx->capturing) c->halo_updates++;
    ctx->launches++;
    return 0;
}

int hemo_comm_allreduce_j(hemo_ctx* ctx, double* buf, int count) {
    HemoComm* c = ctx->comm;
    if (!c || c->nranks == 1) return 0;
    HEMO_PROF_BEGIN(ctx, HEMO_PROF_ALLREDUCE);
    HEMO_CHECK_NCCL(ctx, g_nccl.AllReduce(buf, buf, (size_t)count, ncclFloat64, ncclSum, c->comm, ctx->stream));
    HEMO_PROF_END(ctx, HEMO_PROF_ALLREDUCE);
    if (!ctx->capturing) c->allreduces++;
    ctx->launches++;
    return 0;
}

extern "C" int hemo_comm_halo_update(hemo_ctx* ctx, double* v_dev) {
    if (!ctx || !v_dev) return HEMO_EINVAL;
    if (!ctx->comm) HEMO_FAIL(ctx, HEMO_ESTATE, "no communicator (hemo_comm_init)");
    return hemo_comm_halo(ctx, v_dev);
}

extern "C" int hemo_comm_allreduce(hemo_ctx* ctx, double* buf_dev, int count) {
    if (!ctx || !buf_dev || count < 1) return HEMO_EINVAL;
    if (!ctx->comm) HEMO_FAIL(ctx, HEMO_ESTATE, "no communicator (hemo_comm_init)");
    return hemo_comm_allreduce_j(ctx, buf_dev, count);
}
