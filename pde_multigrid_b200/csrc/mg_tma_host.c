/*
 * mg_tma_host.c -- host-side creation of TMA tensor maps (CUtensorMap) for the colour-split 3D fields.
 * cuTensorMapEncodeTiled is a driver-API call; it is resolved through cudaGetDriverEntryPoint so the
 * library does not link against libcuda directly.
 */
#include <cuda.h>
#include <string.h>

#include "mg_host_common.h"

typedef CUresult (*encode_tiled_fn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                    const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                    CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static encode_tiled_fn g_encode = NULL;

static int resolve(void)
{
    if (g_encode) return MG_OK;
    void* fn = NULL;
    enum cudaDriverEntryPointQueryResult q;
    cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q);
    if (e != cudaSuccess || q != cudaDriverEntryPointSuccess || !fn)
        return mg_fail(MG_ERR_CUDA, "cuTensorMapEncodeTiled is not available from this driver (%s)", cudaGetErrorString(e));
    g_encode = (encode_tiled_fn)fn;
    return MG_OK;
}

/* One colour array of a colour-split field as a rank-3 tensor (hp, n, nzl) with a (box_i, box_y, 1) box.
   out128 receives the 128-byte CUtensorMap. */
int mg_tma_make_colour_map(void* out128, int dtype, void* base, const mg_geom3d* g, int box_i, int box_y)
{
    int st = resolve();
    if (st) return st;
    const size_t es = mg_esize(dtype);
    cuuint64_t dims[3] = {(cuuint64_t)g->hp, (cuuint64_t)g->n, (cuuint64_t)g->nzl};
    cuuint64_t strides[2] = {(cuuint64_t)g->hp * es, (cuuint64_t)g->plane * es};
    cuuint32_t box[3] = {(cuuint32_t)box_i, (cuuint32_t)box_y, 1};
    cuuint32_t estr[3] = {1, 1, 1};
    CUtensorMap map;
    CUresult r = g_encode(&map, dtype == MG_F32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 3, base, dims,
                          strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                          CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return mg_fail(MG_ERR_CUDA, "cuTensorMapEncodeTiled failed with CUresult %d (hp=%d n=%d nzl=%d box=%dx%d)", (int)r, g->hp, g->n, g->nzl, box_i, box_y);
    memcpy(out128, &map, sizeof map);
    return MG_OK;
}
