/* mg_comm.c -- see mg_comm.h */
#include "mg_comm.h"

#include <dlfcn.h>
#include <nccl.h>
#include <stdlib.h>
#include <string.h>

struct mg_comm_s {
    ncclComm_t comm;
    int rank;
};

static struct {
    void* lib;
    ncclResult_t (*GetUniqueId)(ncclUniqueId*);
    ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int);
    ncclResult_t (*CommDestroy)(ncclComm_t);
    ncclResult_t (*Send)(const void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t);
    ncclResult_t (*Recv)(void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t);
    ncclResult_t (*GroupStart)(void);
    ncclResult_t (*GroupEnd)(void);
    ncclResult_t (*AllReduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t);
    ncclResult_t (*AllGather)(const void*, void*, size_t, ncclDataType_t, ncclComm_t, cudaStream_t);
    const char* (*GetErrorString)(ncclResult_t);
} N;

static int nccl_load(void)
{
    if (N.lib) return MG_OK;
    void* h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
    if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
    if (!h) return mg_fail(MG_ERR_COMM, "cannot load libnccl.so.2: %s", dlerror());
#define SYM(field, name)                                                                       \
    do {                                                                                       \
        *(void**)(&N.field) = dlsym(h, name);                                                  \
        if (!N.field) return mg_fail(MG_ERR_COMM, "libnccl.so.2 lacks the symbol %s", name);   \
    } while (0)
    SYM(GetUniqueId, "ncclGetUniqueId");
    SYM(CommInitRank, "ncclCommInitRank");
    SYM(CommDestroy, "ncclCommDestroy");
    SYM(Send, "ncclSend");
    SYM(Recv, "ncclRecv");
    SYM(GroupStart, "ncclGroupStart");
    SYM(GroupEnd, "ncclGroupEnd");
    SYM(AllReduce, "ncclAllReduce");
    SYM(AllGather, "ncclAllGather");
    SYM(GetErrorString, "ncclGetErrorString");
#undef SYM
    N.lib = h;
    return MG_OK;
}

#define MG_NCCL(call)                                                                                      \
    do {                                                                                                   \
        ncclResult_t r_ = (call);                                                                          \
        if (r_ != ncclSuccess) return mg_fail(MG_ERR_COMM, "%s failed: %s", #call, N.GetErrorString(r_));  \
    } while (0)

static ncclDataType_t nccl_type(int dtype) { return dtype == MG_F32 ? ncclFloat32 : ncclFloat64; }

int mg_comm_unique_id(void* out128)
{
    if (!out128) return mg_fail(MG_ERR_ARG, "null argument");
    int st = nccl_load();
    if (st) return st;
    ncclUniqueId id;
    MG_NCCL(N.GetUniqueId(&id));
    memcpy(out128, &id, sizeof id < 128 ? sizeof id : 128);
    return MG_OK;
}

int mg_comm_create(mg_comm** out, int rank, int nranks, const void* unique_id128)
{
    if (!out || !unique_id128 || nranks < 1 || rank < 0 || rank >= nranks) return mg_fail(MG_ERR_ARG, "bad communicator arguments");
    int st = nccl_load();
    if (st) return st;
    mg_comm* c = (mg_comm*)calloc(1, sizeof *c);
    if (!c) return mg_fail(MG_ERR_NOMEM, "host allocation failed");
    ncclUniqueId id;
    memset(&id, 0, sizeof id);
    memcpy(&id, unique_id128, sizeof id < 128 ? sizeof id : 128);
    ncclResult_t r = N.CommInitRank(&c->comm, nranks, id, rank);
    if (r != ncclSuccess) {
        free(c);
        return mg_fail(MG_ERR_COMM, "ncclCommInitRank failed: %s", N.GetErrorString(r));
    }
    c->rank = rank;
    *out = c;
    return MG_OK;
}

void mg_comm_destroy(mg_comm* c)
{
    if (!c) return;
    if (c->comm) N.CommDestroy(c->comm);
    free(c);
}

int mg_comm_group_start(mg_comm* c) { (void)c; MG_NCCL(N.GroupStart()); return MG_OK; }
int mg_comm_group_end(mg_comm* c) { (void)c; MG_NCCL(N.GroupEnd()); return MG_OK; }

int mg_comm_send(mg_comm* c, const void* buf, size_t count, int dtype, int peer, cudaStream_t s)
{
    MG_NCCL(N.Send(buf, count, nccl_type(dtype), peer, c->comm, s));
    return MG_OK;
}

int mg_comm_recv(mg_comm* c, void* buf, size_t count, int dtype, int peer, cudaStream_t s)
{
    MG_NCCL(N.Recv(buf, count, nccl_type(dtype), peer, c->comm, s));
    return MG_OK;
}

int mg_comm_allreduce_sum_max(mg_comm* c, double* buf2, cudaStream_t s)
{
    MG_NCCL(N.GroupStart());
    MG_NCCL(N.AllReduce(buf2, buf2, 1, ncclFloat64, ncclSum, c->comm, s));
    MG_NCCL(N.AllReduce(buf2 + 1, buf2 + 1, 1, ncclFloat64, ncclMax, c->comm, s));
    MG_NCCL(N.GroupEnd());
    return MG_OK;
}

int mg_comm_allreduce_u64_sum(mg_comm* c, unsigned long long* buf1, cudaStream_t s)
{
    MG_NCCL(N.AllReduce(buf1, buf1, 1, ncclUint64, ncclSum, c->comm, s));
    return MG_OK;
}

int mg_comm_allgather_inplace(mg_comm* c, void* recvbuf, size_t count, int dtype, cudaStream_t s)
{
    const char* send = (const char*)recvbuf + (size_t)c->rank * count * mg_esize(dtype);
    MG_NCCL(N.AllGather(send, recvbuf, count, nccl_type(dtype), c->comm, s));
    return MG_OK;
}
