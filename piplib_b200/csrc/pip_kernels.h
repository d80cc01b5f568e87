/* internal launch interface between the host layer (pip_host.cpp) and the kernels */
#ifndef PIP_KERNELS_H
#define PIP_KERNELS_H

#include <cuda_runtime.h>

#include "pip_convert.h"
#include "pip_types.h"

#define PIP_WARPS_PER_CTA_MAX 4
#define PIP_CTA_THREADS (PIP_WARPS_PER_CTA_MAX * 32)
#ifndef PIP_MIN_CTAS
#define PIP_MIN_CTAS 4      /* <= 128 registers per thread */
#endif

#ifdef __cplusplus
extern "C" {
#endif
cudaError_t pip_launch_solve(const PipLaunch *L, int shared_class, int ctas, int warps_per_cta, cudaStream_t stream);
cudaError_t pip_solve_occupancy(int shared_class, int warps_per_cta, size_t smem_bytes, int *ctas_per_sm);
cudaError_t pip_launch_gather(PipResult *res, const int *order, const PipCell *cells, long long *dst_off,
                              pip_u64 *out, int nprob, long long *total, int phase, cudaStream_t stream);
/* pass 0: size the streams the solver did not size; pass 1: decode (parm per problem, or *uparm for all;
 * placement by dst_off, or by span reservation when so != NULL) */
cudaError_t pip_launch_serialize(PipResult *res, const int *order, const PipCell *cells, const PipDecodeParm *parm,
                                 const PipDecodeParm *uparm, const long long *dst_off, pip_i64 *out, pip_u64 *hashes,
                                 int nprob, int pass, const PipStreamOut *so, cudaStream_t stream);
/* word mode: copy the streams the solver wrote itself into the compact buffer (span reservation) */
cudaError_t pip_launch_gather_words(PipResult *res, const int *order, const PipCell *cells, pip_i64 *out,
                                    int nprob, const PipStreamOut *so, const PipSteal *stl, int sol_size,
                                    cudaStream_t stream);
cudaError_t pip_launch_init_results(PipResult *res, long long n, cudaStream_t stream);
cudaError_t pip_launch_convert(const PipConvertArgs *A, int elem_log2, cudaStream_t stream);
/* a stream_out chunk's per-problem arrays (PipDeviceOut) -> the caller's device arrays at the chunk's first problem;
 * hashes / ser_off / ser_len / info may be NULL (info needs the chunk's reports `inf`) */
cudaError_t pip_launch_emit_device(const int *st, const pip_u64 *hs, const long long *off, const long long *len,
                                   const PipInfo *inf, long long n, long long base, int *status, pip_u64 *hashes,
                                   long long *ser_off, long long *ser_len, PipInfo *info, cudaStream_t stream);
cudaError_t pip_launch_image(const PipProblem *prob, const void *pool, int elem_log2, long long n, const PipLayout *lay,
                             pip_i64 *images, int image_words, int image_w1, int vbytes, cudaStream_t stream);
int pip_layout_compute(int nvar, int nparm, int ni, int nc, int flags, int level, int words, int vbytes, PipLayout *out);
long long pip_layout_words(int nvar, int nparm, int ni, int nc, int flags, int level, int vbytes);
#ifdef __cplusplus
}
#endif
#endif
