/*
 * mg_comm.h -- thin NCCL layer of the multi-GPU (z-slab) 3D driver: one process per GPU, halo planes by
 * grouped ncclSend/ncclRecv on the handle's stream, norms by ncclAllReduce, coarse-level agglomeration by
 * ncclAllGather.  libnccl.so.2 is resolved with dlopen at first use, so the single-GPU library has no
 * NCCL dependency and, inside a torchrun process, the NCCL that torch already loaded is reused.
 */
#ifndef MG_COMM_H
#define MG_COMM_H

#include "mg_host_common.h"

typedef struct mg_comm_s mg_comm;

int mg_comm_create(mg_comm** out, int rank, int nranks, const void* unique_id128);
void mg_comm_destroy(mg_comm* c);

int mg_comm_group_start(mg_comm* c);
int mg_comm_group_end(mg_comm* c);
int mg_comm_send(mg_comm* c, const void* buf, size_t count, int dtype, int peer, cudaStream_t s);
int mg_comm_recv(mg_comm* c, void* buf, size_t count, int dtype, int peer, cudaStream_t s);
/* in-place on device doubles: buf[0] summed, buf[1] maximised over the ranks */
int mg_comm_allreduce_sum_max(mg_comm* c, double* buf2, cudaStream_t s);
/* in-place on one device uint64: summed (mod 2^64) over the ranks */
int mg_comm_allreduce_u64_sum(mg_comm* c, unsigned long long* buf1, cudaStream_t s);
/* in-place all-gather: every rank contributes `count` elements located at recvbuf + rank*count */
int mg_comm_allgather_inplace(mg_comm* c, void* recvbuf, size_t count, int dtype, cudaStream_t s);

#endif
