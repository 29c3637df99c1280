/*
 * mg_profile.h -- per-level, per-operator device timers shared by the host drivers: CUDA event pairs
 * recorded on the handle's stream around operator calls, read back after a synchronise.  Gives the
 * live per-kernel durations bench.py uses for the roofline (events see exactly the stream the kernels
 * are launched on).
 */
#ifndef MG_PROFILE_H
#define MG_PROFILE_H

#include <cuda_runtime_api.h>

#include "../../include/mg_b200.h"

#define MG_PROF_MAX_LEVELS 32

typedef struct {
    int enabled;
    int n, cap;          /* recorded pairs */
    cudaEvent_t* ev;     /* 2 per pair */
    int* level;
    int* op;
    long long* launches; /* kernels launched inside the pair */
    long long open_launches;
    double ms[MG_PROF_MAX_LEVELS][MG_OP_COUNT];
    long long kl[MG_PROF_MAX_LEVELS][MG_OP_COUNT];
    long long calls[MG_PROF_MAX_LEVELS][MG_OP_COUNT];
} mg_prof;

int mg_prof_enable(mg_prof* p, cudaStream_t s, int enable);
void mg_prof_begin(mg_prof* p, cudaStream_t s, int level, int op, long long launches_now);
void mg_prof_end(mg_prof* p, cudaStream_t s, long long launches_now);
int mg_prof_collect(mg_prof* p, cudaStream_t s); /* synchronises, folds recorded pairs into the tables */
void mg_prof_free(mg_prof* p);

#endif
