/* mg_profile.c -- see mg_profile.h */
#include "mg_host_common.h"

#include <stdlib.h>
#include <string.h>

int mg_prof_enable(mg_prof* p, cudaStream_t s, int enable)
{
    if (enable) {
        int st = mg_prof_collect(p, s);
        if (st) return st;
        memset(p->ms, 0, sizeof p->ms);
        memset(p->kl, 0, sizeof p->kl);
        memset(p->calls, 0, sizeof p->calls);
    }
    p->enabled = enable != 0;
    return MG_OK;
}

void mg_prof_begin(mg_prof* p, cudaStream_t s, int level, int op, long long launches_now)
{
    if (!p->enabled) return;
    if (p->n == p->cap) {
        int ncap = p->cap ? 2 * p->cap : 256;
        p->ev = (cudaEvent_t*)realloc(p->ev, 2 * (size_t)ncap * sizeof(cudaEvent_t));
        p->level = (int*)realloc(p->level, (size_t)ncap * sizeof(int));
        p->op = (int*)realloc(p->op, (size_t)ncap * sizeof(int));
        p->launches = (long long*)realloc(p->launches, (size_t)ncap * sizeof(long long));
        for (int i = p->cap; i < ncap; i++) {
            cudaEventCreate(&p->ev[2 * i]);
            cudaEventCreate(&p->ev[2 * i + 1]);
        }
        p->cap = ncap;
    }
    p->level[p->n] = level < MG_PROF_MAX_LEVELS ? level : MG_PROF_MAX_LEVELS - 1;
    p->op[p->n] = op;
    p->open_launches = launches_now;
    cudaEventRecord(p->ev[2 * p->n], s);
}

void mg_prof_end(mg_prof* p, cudaStream_t s, long long launches_now)
{
    if (!p->enabled) return;
    cudaEventRecord(p->ev[2 * p->n + 1], s);
    p->launches[p->n] = launches_now - p->open_launches;
    p->n++;
}

int mg_prof_collect(mg_prof* p, cudaStream_t s)
{
    if (p->n == 0) return MG_OK;
    MG_CUDA(cudaStreamSynchronize(s));
    for (int i = 0; i < p->n; i++) {
        float ms = 0.f;
        MG_CUDA(cudaEventElapsedTime(&ms, p->ev[2 * i], p->ev[2 * i + 1]));
        p->ms[p->level[i]][p->op[i]] += ms;
        p->kl[p->level[i]][p->op[i]] += p->launches[i];
        p->calls[p->level[i]][p->op[i]] += 1;
    }
    p->n = 0;
    return MG_OK;
}

void mg_prof_free(mg_prof* p)
{
    for (int i = 0; i < 2 * p->cap; i++) cudaEventDestroy(p->ev[i]);
    free(p->ev); free(p->level); free(p->op); free(p->launches);
    memset(p, 0, sizeof *p);
}
