/* sm_100a kernels of the batched PipLib solver core and their launch wrappers.
 *
 *   pip_solve_kernel<true>   size class S: one problem per warp, working set in shared memory
 *   pip_solve_kernel<false>  size class G: one problem per warp, working set in global memory
 *                            (L1/L2 resident; for tableaus that outgrow a shared-memory arena)
 *   pip_gather_kernel        compacts the per-warp cell windows into one contiguous stream in
 *                            problem order, so the device-to-host copy is a single memcpy
 *   pip_scan kernels         exclusive scan of the per-problem cell counts
 */
#include <cuda_runtime.h>
#include <stdint.h>

#include <stdlib.h>
#include <string.h>

#include <mutex>

#include "pip_convert.h"
#include "pip_decode.h"
#include "pip_decode_warp.h"
#include "pip_kernels.h"
#include "pip_segments.h"
#include "pip_warp_main.h"

extern __shared__ __align__(16) unsigned char pip_smem[];

/* cudaFuncAttributeMaxDynamicSharedMemorySize is process-wide per kernel while launches come from
 * several engine lanes at once: the limit is only ever raised, under one lock, so that no lane can
 * lower it between another lane's query and its launch */
static std::mutex g_attr_mu;
template <class K>
static cudaError_t pip_raise_dynamic_smem(K kernel, size_t bytes, size_t &high_water)
{
  std::lock_guard<std::mutex> g(g_attr_mu);
  if (bytes <= high_water) return cudaSuccess;
  cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
  if (e == cudaSuccess) high_water = bytes;
  return e;
}
static size_t g_smem_s32 = 0, g_smem_s64 = 0, g_smem_ws = 0, g_smem_team = 0, g_smem_s32_steal = 0, g_smem_s64_steal = 0;

template <bool SH, class V, bool STEAL = false, bool WORDS = false>
__global__ void __launch_bounds__(PIP_CTA_THREADS, PIP_MIN_CTAS)
pip_solve_kernel(const PipLaunch L)
{
  const int warp_in_cta = threadIdx.x >> 5;
  const int warps_per_cta = blockDim.x >> 5;
  const int warp_id = blockIdx.x * warps_per_cta + warp_in_cta;
  pip_i64 *arena;
  if (SH) arena = (pip_i64 *)pip_smem + (size_t)warp_in_cta * L.work_words;
  else arena = L.gwork + (size_t)warp_id * L.work_words;
  pip_warp_main<V, !SH, STEAL, WORDS>(L, warp_id, arena, nullptr);   /* !SH: the global-memory code path */
}

/* size class M: one problem per CTA, arena in global memory.  Warp 0 runs the solver, the other
 * warps join it for the rank-1 update of every pivot on a tall tableau (pip_solver.h, PipTeam). */
__global__ void __launch_bounds__(512, 1)
pip_team_kernel(const PipLaunch L)
{
  __shared__ PipTeam team;
  const int tid = threadIdx.x;
  if (tid == 0) { team.nthreads = blockDim.x; team.cmd = PIP_TEAM_UPDATE; team.fault = 0; team.ovf = 0; }
  __syncthreads();
  /* the problem's arena: global memory, or -- when the class's working set fits (pip_engine.cpp) -- the
   * CTA's dynamic shared memory: the tall tableaus of cut chains (vivien32: 303 rows x 23 words = 56 KB)
   * then never leave the SM */
  pip_i64 *arena = L.gwork ? L.gwork + (size_t)blockIdx.x * L.work_words : (pip_i64 *)pip_smem;
  if (tid < 32) {
    pip_warp_main<pip_i64, true>(L, blockIdx.x, arena, &team);
    if (tid == 0) team.cmd = PIP_TEAM_EXIT;
    __syncwarp();
    pip_team_barrier(team.nthreads);
  } else pip_team_helper<pip_i64>(&team, tid);
}

/* shared_class: 0 = global-memory arena (int64), 1 = shared arena int64, 2 = shared arena int32,
 * 3 = team (class M): `warps_per_cta` warps work on one problem, `ctas` problems in flight; 4 = team with the
 * arena in shared memory (L->gwork == NULL, work_words * 8 bytes of dynamic shared memory per CTA) */
extern "C" cudaError_t pip_launch_solve(const PipLaunch *L, int shared_class, int ctas, int warps_per_cta,
                                        cudaStream_t stream)
{
  if (shared_class == 1 || shared_class == 2) {
    size_t smem = (size_t)warps_per_cta * L->work_words * sizeof(pip_i64);
    cudaError_t e;
    /* subtree donation (PipLaunch::steal) runs the instantiation that has it compiled in (word mode only);
     * word-mode launches the one without the cell emitters */
#define PIP_LAUNCH_S(V_, ST_, WD_, hw_) do { \
      e = pip_raise_dynamic_smem(pip_solve_kernel<true, V_, ST_, WD_>, smem, hw_); \
      if (e != cudaSuccess) return e; \
      pip_solve_kernel<true, V_, ST_, WD_><<<ctas, warps_per_cta * 32, smem, stream>>>(*L); } while (0)
    static size_t hw_words32 = 0, hw_words64 = 0;
    const bool words = L->emit_words != 0;
    if (L->steal.mode && !words) return cudaErrorInvalidValue;
    if (shared_class == 2 && L->steal.mode) PIP_LAUNCH_S(int, true, true, g_smem_s32_steal);
    else if (shared_class == 2 && words) PIP_LAUNCH_S(int, false, true, hw_words32);
    else if (shared_class == 2) PIP_LAUNCH_S(int, false, false, g_smem_s32);
    else if (L->steal.mode) PIP_LAUNCH_S(pip_i64, true, true, g_smem_s64_steal);
    else if (words) PIP_LAUNCH_S(pip_i64, false, true, hw_words64);
    else PIP_LAUNCH_S(pip_i64, false, false, g_smem_s64);
#undef PIP_LAUNCH_S
  } else if (shared_class == 4) {
    const size_t smem = (size_t)L->work_words * sizeof(pip_i64);
    cudaError_t e = pip_raise_dynamic_smem(pip_team_kernel, smem, g_smem_team);
    if (e != cudaSuccess) return e;
    pip_team_kernel<<<ctas, warps_per_cta * 32, smem, stream>>>(*L);
  } else if (shared_class == 3) {
    pip_team_kernel<<<ctas, warps_per_cta * 32, 0, stream>>>(*L);
  } else {
    pip_solve_kernel<false, pip_i64><<<ctas, warps_per_cta * 32, 0, stream>>>(*L);
  }
  return cudaGetLastError();
}

extern "C" cudaError_t pip_solve_occupancy(int shared_class, int warps_per_cta, size_t smem_bytes, int *ctas_per_sm)
{
  if (shared_class == 4) {
    cudaError_t e = pip_raise_dynamic_smem(pip_team_kernel, smem_bytes, g_smem_team);
    if (e != cudaSuccess) return e;
    return cudaOccupancyMaxActiveBlocksPerMultiprocessor(ctas_per_sm, pip_team_kernel, warps_per_cta * 32, smem_bytes);
  }
  if (shared_class == 2) {
    cudaError_t e = pip_raise_dynamic_smem(pip_solve_kernel<true, int>, smem_bytes, g_smem_s32);
    if (e != cudaSuccess) return e;
    return cudaOccupancyMaxActiveBlocksPerMultiprocessor(ctas_per_sm, pip_solve_kernel<true, int>, warps_per_cta * 32, smem_bytes);
  }
  if (shared_class) {
    cudaError_t e = pip_raise_dynamic_smem(pip_solve_kernel<true, pip_i64>, smem_bytes, g_smem_s64);
    if (e != cudaSuccess) return e;
    return cudaOccupancyMaxActiveBlocksPerMultiprocessor(ctas_per_sm, pip_solve_kernel<true, pip_i64>, warps_per_cta * 32, smem_bytes);
  }
  return cudaOccupancyMaxActiveBlocksPerMultiprocessor(ctas_per_sm, pip_solve_kernel<false, pip_i64>, warps_per_cta * 32, 0);
}

/* words of working arena a problem needs at a slack level (host-side planning) */
extern "C" long long pip_layout_words(int nvar, int nparm, int ni, int nc, int flags, int level, int vbytes)
{
  PipLayout L;
  pip_layout(nvar, nparm, ni, nc, flags, level, 0x7fffffff, vbytes, L);
  return L.total;
}

/* ---- arena images (dense batches): the problem load of the solver, run ahead of it ----------------------
 * One warp per problem runs the solver's own loader (pip_load_problem: element widening, den / fl, tab_simplify)
 * into the problem's image in global memory, laid out like the arena regions it stands for (offsets rebased to
 * the image).  The solve kernel then starts every problem with two block copies, and the loader -- 270
 * instructions that ran once per problem -- is out of its instruction stream (DESIGN.md section 4). */
template <class V>
__global__ void __launch_bounds__(256) pip_image_kernel(const PipProblem *prob, const void *pool, int elem_log2, long long n,
                                                        const PipLayout lay, pip_i64 *images, int image_words, int image_w1)
{
  const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
  PipLayout L = lay;
  L.m.fl -= L.m.den; L.tmp -= L.m.den; L.m.data -= L.m.den; L.m.den = 0;
  L.ctx = image_w1;
  for (long long p = warp; p < n; p += nwarps) {
    const PipProblem P = prob[p];
    if (P.flags & PIP_F_WIDE_INPUT) continue;            /* solved from the int64 pool by the general loader */
    L.m.ni = P.ni;
    PipSolver<V>::pip_load_problem(P, pool, elem_log2, images + p * image_words, L.m, L.ctx, L.cstride);
  }
}

extern "C" cudaError_t pip_launch_image(const PipProblem *prob, const void *pool, int elem_log2, long long n, const PipLayout *lay,
                                        pip_i64 *images, int image_words, int image_w1, int vbytes, cudaStream_t stream)
{
  long long blocks = (n + 7) / 8;
  if (blocks > 148 * 16) blocks = 148 * 16;
  if (blocks < 1) blocks = 1;
  if (vbytes == 4) pip_image_kernel<int><<<(int)blocks, 256, 0, stream>>>(prob, pool, elem_log2, n, *lay, images, image_words, image_w1);
  else pip_image_kernel<pip_i64><<<(int)blocks, 256, 0, stream>>>(prob, pool, elem_log2, n, *lay, images, image_words, image_w1);
  return cudaGetLastError();
}

/* the arena layout of a shape at a slack level, degraded exactly as the solver degrades it when the arena is
 * too small; out->s.ni carries nc + 1 (the largest context the layout was carved for).  0 = does not fit */
extern "C" int pip_layout_compute(int nvar, int nparm, int ni, int nc, int flags, int level, int words, int vbytes,
                                  PipLayout *out)
{
  int level_try = level;
  while (!pip_layout(nvar, nparm, ni, nc, flags, level_try, words, vbytes, *out)) {
    level_try = level_try == PIP_LEVEL_S_WIDE ? 2 : level_try - 1;
    if (level_try < 0) return 0;
  }
  out->s.ni = nc + 1;
  return 1;
}

/* ---- cell gather ------------------------------------------------------------------------ */
/* one warp per problem: move its cells from the warp windows to the compact word stream at
 * dst_off[q], packing each cell into one word unless the problem is flagged wide */
__global__ void pip_gather_kernel(PipResult *res, const int *order, const PipCell *cells,
                                  const long long *dst_off, pip_u64 *out, int nprob)
{
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  const int nwarps = (gridDim.x * blockDim.x) >> 5;
  for (int q = warp; q < nprob; q += nwarps) {
    const int p = order ? order[q] : q;
    const PipResult r = res[p];
    const PipCell *src = cells + r.cell_off;
    pip_u64 *dst = out + dst_off[q];
    if (r.rflags & PIP_RES_WIDE) {
      const pip_u64 *s3 = (const pip_u64 *)src;
      for (int w = lane; w < r.ncells * 3; w += 32) dst[w] = s3[w];
    } else {
      for (int c = lane; c < r.ncells; c += 32) dst[c] = PIP_CELL_PACK(src[c].kind, src[c].p1, src[c].p2);
    }
    __syncwarp();
    if (lane == 0) res[p].cell_off = dst_off[q];      /* now a word offset into the compact stream */
  }
}

/* ---- device-side decode: cells -> serialised quast words (pip_decode.h) --------------------- */
/* sizing pass, one thread per problem, for streams the solver did not size itself (column surgery:
 * Maximize / Urs_* / a big parameter): words of the stream, and whether they fit int32 */
__global__ void pip_serialize_kernel(PipResult *res, const int *order, const PipCell *cells,
                                     const PipDecodeParm *parm, const PipDecodeParm uparm, int nprob)
{
  const int q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= nprob) return;
  const int p = order ? order[q] : q;
  const PipResult r = res[p];
  PipSer s;
  s.out = nullptr; s.cap = 0;
  s.len = 0; s.h = PIP_HASH_INIT; s.hashing = 0; s.narrow_out = 0; s.wide = 0;
  if (r.status == PIP_ST_VOID) pip_sput(s, -1);
  else if (r.status == PIP_ST_OK) {
    PipRawCells c = {cells + r.cell_off};
    const PipDecodeParm d = parm ? parm[p] : uparm;
    pip_ser_cells(s, c, r.ncells, d.bg, d.urs, d.flags);
  }
  res[p].ser_words = (unsigned)s.len;
  if (!s.wide) res[p].rflags = r.rflags | PIP_RES_SER32;
}

/* pass 1 with one warp per problem (pip_decode_warp.h): cells staged in shared memory by a coalesced
 * copy, warp-uniform parse, lane-parallel vectors, words out through a hashed shared-memory tile.
 * Two ways to place the output: `dst_off` (an exclusive scan computed beforehand, cell-gather path) or
 * `so.ctl` (dense path): the warp reserves the span with one atomic add, writes the per-problem results
 * in structure-of-arrays form and sums the counters of finished problems. */
#define PIP_WS_WARPS 8
#define PIP_WS_WORDS_PER_WARP (PIP_WS_TILE + 3 * PIP_WS_CELLS)
__global__ void __launch_bounds__(32 * PIP_WS_WARPS)
pip_serialize_warp_kernel(PipResult *res, const int *order, const PipCell *cells, const PipDecodeParm *parm,
                          const PipDecodeParm uparm, const long long *dst_off, pip_i64 *out, pip_u64 *hashes, int nprob,
                          const PipStreamOut so)
{
  const int wid = threadIdx.x >> 5, lane = threadIdx.x & 31;
  pip_i64 *tile = (pip_i64 *)pip_smem + (size_t)wid * PIP_WS_WORDS_PER_WARP;
  pip_i64 *stage = tile + PIP_WS_TILE;
  const bool stream = so.ctl != nullptr;
  unsigned long long acc[7] = {0, 0, 0, 0, 0, 0, 0};
  unsigned mrows = 0, mcols = 0, finals = 0;
  for (int q = blockIdx.x * PIP_WS_WARPS + wid; q < nprob; q += gridDim.x * PIP_WS_WARPS) {
    const int p = order ? order[q] : q;
    const PipResult r = res[p];
    const bool narrow = (r.rflags & PIP_RES_SER32) != 0 && !(stream && so.words64);
    PipWarpSer s;
    s.tile = tile; s.cap = (long long)r.ser_words; s.len = 0; s.fill = 0;
    s.h = 0; s.narrow_out = narrow ? 1 : 0; s.wide = 0;
    long long base = 0;
    const bool has_words = r.status == PIP_ST_OK || r.status == PIP_ST_VOID;
    if (stream) {
      const long long slots = !has_words ? 0 : narrow ? ((long long)r.ser_words + 1) / 2 : (long long)r.ser_words;
      if (lane == 0 && slots) base = (long long)atomicAdd(so.ctl + PIP_SO_SLOTS, (unsigned long long)slots);
      base = __shfl_sync(0xffffffffu, base, 0);
      s.out = out + base;
      if (base + slots > so.cap) {                     /* does not fit: count only, the host grows the buffer */
        s.out = nullptr;
        if (lane == 0) so.ctl[PIP_SO_OVERFLOW] = 1;
      }
    } else { base = dst_off[q]; s.out = out + base; }
    if (r.status == PIP_ST_VOID) pip_wput(s, -1);
    else if (r.status == PIP_ST_OK) {
      const PipCell *src = cells + r.cell_off;
      if (r.ncells <= PIP_WS_CELLS) {
        const pip_i64 *g = (const pip_i64 *)src;
        for (int k = lane; k < 3 * (int)r.ncells; k += 32) stage[k] = g[k];
        __syncwarp();
        src = (const PipCell *)stage;
      }
      PipRawCells c = {src};
      const PipDecodeParm d = parm ? parm[p] : uparm;
      pip_wser_cells(s, c, r.ncells, d.bg, d.urs, d.flags);
    }
    pip_wser_flush(s);
    const pip_u64 hsum = pip_wser_hash(s);
    /* a stream sized by the solver (PIP_RES_SIZED) must come out exactly that long and, when it was
     * promised narrow, fit 32-bit words: anything else is a bug, never a silent truncation */
    const bool bad = (r.rflags & PIP_RES_SIZED) && has_words && (s.len != (long long)r.ser_words || (narrow && s.wide));
    if (lane == 0) {
      const pip_u64 h = has_words ? hsum : 0ull;
      if (stream) {
        so.status[p] = bad ? PIP_ST_FAULT + 1 : r.status;
        so.hash[p] = h;
        so.off[p] = base;
        so.len[p] = has_words ? ((long long)r.ser_words | (narrow ? PIP_LEN_NARROW : 0ll)) : 0ll;
        if (so.info) so.info[p] = pip_info_of(r);
      } else {
        res[p].cell_off = base;
        if (hashes) hashes[p] = h;
        if (bad) res[p].status = PIP_ST_FAULT + 1;
      }
    }
    if (stream && PIP_STATUS_IS_FINAL(r.status)) {
      finals++;
      acc[0] += r.pivots; acc[1] += r.cuts; acc[2] += r.subsolves; acc[3] += r.splits;
      acc[4] += ((unsigned long long)r.elem_updates_hi << 32) | r.elem_updates_lo;
      acc[5] += (unsigned long long)r.ncells;
      acc[6] += (r.rflags & PIP_RES_WRAPPED) ? 1ull : 0ull;
      mrows = r.max_rows > mrows ? r.max_rows : mrows;
      mcols = r.max_cols > mcols ? r.max_cols : mcols;
    }
    __syncwarp();
  }
  if (stream && lane == 0 && finals) {
    atomicAdd(so.ctl + PIP_SO_FINALS, (unsigned long long)finals);
    for (int k = 0; k < 6; k++) atomicAdd(so.stats + k, acc[k]);
    atomicMax(so.stats + 6, (unsigned long long)mrows);
    atomicMax(so.stats + 7, (unsigned long long)mcols);
    if (acc[6]) atomicAdd(so.stats + 8, acc[6]);
  }
}

extern "C" cudaError_t pip_launch_serialize(PipResult *res, const int *order, const PipCell *cells,
                                            const PipDecodeParm *parm, const PipDecodeParm *uparm,
                                            const long long *dst_off, pip_i64 *out,
                                            pip_u64 *hashes, int nprob, int pass, const PipStreamOut *so,
                                            cudaStream_t stream)
{
  PipDecodeParm u = {0, 0, 0};
  if (uparm) u = *uparm;
  if (pass == 1) {
    PipStreamOut o;
    memset(&o, 0, sizeof o);
    if (so) o = *so;
    const size_t smem = sizeof(pip_i64) * PIP_WS_WARPS * PIP_WS_WORDS_PER_WARP;
    cudaError_t e = pip_raise_dynamic_smem(pip_serialize_warp_kernel, smem, g_smem_ws);
    if (e != cudaSuccess) return e;
    int blocks = (nprob + PIP_WS_WARPS - 1) / PIP_WS_WARPS;
    if (blocks > 148 * 3) blocks = 148 * 3;
    pip_serialize_warp_kernel<<<blocks, 32 * PIP_WS_WARPS, smem, stream>>>(res, order, cells, parm, u, dst_off, out, hashes,
                                                                          nprob, o);
    return cudaGetLastError();
  }
  const int threads = 128;
  pip_serialize_kernel<<<(nprob + threads - 1) / threads, threads, 0, stream>>>(res, order, cells, parm, u, nprob);
  return cudaGetLastError();
}

/* word mode (the solver wrote the serialised quast itself): what is left of the decode is a copy -- reserve the
 * problem's span of the compact buffer, move the words (int32 from class S32, int64 otherwise; written as
 * int32 or int64 as the caller asked), fill the per-problem arrays, sum the counters.  One warp per problem. */
__global__ void __launch_bounds__(256)
pip_gather_words_kernel(PipResult *res, const int *order, const PipCell *cells, pip_i64 *out, int nprob,
                        const PipStreamOut so, const PipSteal stl, int sol_size)
{
  const int lane = threadIdx.x & 31;
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = (gridDim.x * blockDim.x) >> 5;
  unsigned long long acc[7] = {0, 0, 0, 0, 0, 0, 0};
  unsigned mrows = 0, mcols = 0, finals = 0;
  for (int q = warp; q < nprob; q += nwarps) {
    const int p = order ? order[q] : q;
    PipResult r = res[p];
    /* subtrees of this problem solved by other warps (PipSteal): resolve the verdict over the segment list */
    const int chain = stl.mode ? stl.head_next[p] : -1;
    PipResolved R;
    if (chain >= 0) {
      pip_resolve_segments(r, chain, stl, sol_size, R);
      r.status = R.status;
      r.ser_words = (unsigned)R.words; r.ncells = (int)R.cells;
      r.pivots = (unsigned)R.pivots; r.cuts = (unsigned)R.cuts; r.subsolves = (unsigned)R.subsolves; r.splits = (unsigned)R.splits;
      r.elem_updates_lo = (unsigned)(R.elem_updates & 0xffffffffull); r.elem_updates_hi = (unsigned)(R.elem_updates >> 32);
      r.max_rows = R.max_rows; r.max_cols = R.max_cols;
      r.rflags = (R.any_flags_or & ~PIP_RES_SER32) | (R.all_flags_and & PIP_RES_SER32);
      /* the reports ask for the counters at the verdict, and a cell limit met inside a donated segment has none
       * (pip_segments.h): such a problem goes back to the ladder, which solves it again without donation */
      if (so.info && r.status == PIP_ST_FATAL + 26 && R.verdict_seg >= 0) r.status = PIP_ST_PENDING;
      if (lane == 0) res[p].status = r.status;         /* the ladder reads the resolved verdict */
    }
    const bool has_words = r.status == PIP_ST_OK || r.status == PIP_ST_VOID;
    const long long nw = has_words ? (long long)r.ser_words : 0;
    const bool narrow = (r.rflags & PIP_RES_SER32) != 0 && !so.words64;
    const long long slots = narrow ? (nw + 1) / 2 : nw;
    long long base = 0;
    if (lane == 0 && slots) base = (long long)atomicAdd(so.ctl + PIP_SO_SLOTS, (unsigned long long)slots);
    base = __shfl_sync(0xffffffffu, base, 0);
    const bool fits = base + slots <= so.cap;          /* else: the host grows the buffer and repeats the pass */
    if (!fits && lane == 0) so.ctl[PIP_SO_OVERFLOW] = 1;
    /* copy and hash in one pass: every lane mixes its own words, the hash is the sum (pip_hash_word); the
     * segments of a problem follow each other in pre-order */
    pip_u64 h = 0;
    if (nw) {
      pip_i64 *dst = out + base;
      long long at = 0;
      int seg = -1;                                       /* -1 = the head segment */
      const bool s32 = (r.rflags & PIP_RES_SRC32) != 0;
      for (;;) {
        const PipResult sr = seg < 0 ? res[p] : stl.segs[seg];
        const void *src = (const void *)(cells + sr.cell_off);
        const long long n = (long long)sr.ser_words;
        for (long long k = lane; k < n; k += 32) {
          const pip_i64 v = s32 ? (pip_i64)((const int *)src)[k] : ((const pip_i64 *)src)[k];
          h += pip_hash_word((pip_u64)v, (pip_u64)(at + k));
          if (fits) { if (narrow) ((int *)dst)[at + k] = (int)v; else dst[at + k] = v; }
        }
        at += n;
        if (chain < 0) break;
        seg = seg < 0 ? chain : stl.seg_next[seg];
        if (seg < 0) break;
      }
    }
    for (int o = 16; o > 0; o >>= 1) h += (pip_u64)__shfl_xor_sync(0xffffffffu, (long long)h, o);
    if (lane == 0) {
      so.status[p] = r.status;
      so.hash[p] = has_words ? h + PIP_HASH_INIT : 0ull;
      so.off[p] = base;
      so.len[p] = nw | (narrow && nw ? PIP_LEN_NARROW : 0ll);
      if (so.info) so.info[p] = pip_info_of(r);
    }
    if (PIP_STATUS_IS_FINAL(r.status)) {
      finals++;
      acc[0] += r.pivots; acc[1] += r.cuts; acc[2] += r.subsolves; acc[3] += r.splits;
      acc[4] += ((unsigned long long)r.elem_updates_hi << 32) | r.elem_updates_lo;
      acc[5] += (unsigned long long)r.ncells;
      acc[6] += (r.rflags & PIP_RES_WRAPPED) ? 1ull : 0ull;
      mrows = r.max_rows > mrows ? r.max_rows : mrows;
      mcols = r.max_cols > mcols ? r.max_cols : mcols;
    }
  }
  if (lane == 0 && finals) {
    atomicAdd(so.ctl + PIP_SO_FINALS, (unsigned long long)finals);
    for (int k = 0; k < 6; k++) atomicAdd(so.stats + k, acc[k]);
    atomicMax(so.stats + 6, (unsigned long long)mrows);
    atomicMax(so.stats + 7, (unsigned long long)mcols);
    if (acc[6]) atomicAdd(so.stats + 8, acc[6]);
  }
}

extern "C" cudaError_t pip_launch_gather_words(PipResult *res, const int *order, const PipCell *cells, pip_i64 *out,
                                               int nprob, const PipStreamOut *so, const PipSteal *stl, int sol_size,
                                               cudaStream_t stream)
{
  int blocks = (nprob + 7) / 8;
  if (blocks > 148 * 8) blocks = 148 * 8;
  if (blocks < 1) blocks = 1;
  PipSteal none;
  memset(&none, 0, sizeof none);
  pip_gather_words_kernel<<<blocks, 256, 0, stream>>>(res, order, cells, out, nprob, *so, stl ? *stl : none, sol_size);
  return cudaGetLastError();
}

/* every record PENDING (the ladder re-arms escalated problems from the host) */
__global__ void pip_init_results_kernel(PipResult *res, long long n)
{
  const long long i0 = (long long)blockIdx.x * blockDim.x + threadIdx.x, step = (long long)gridDim.x * blockDim.x;
  PipResult r;
  memset(&r, 0, sizeof r);
  r.status = PIP_ST_PENDING;
  for (long long i = i0; i < n; i += step) res[i] = r;
}
extern "C" cudaError_t pip_launch_init_results(PipResult *res, long long n, cudaStream_t stream)
{
  int blocks = (int)((n + 255) / 256);
  if (blocks > 148 * 8) blocks = 148 * 8;
  if (blocks < 1) blocks = 1;
  pip_init_results_kernel<<<blocks, 256, 0, stream>>>(res, n);
  return cudaGetLastError();
}

/* ---- device-side input conversion (pip_convert.h): tab_Matrix2Tableau_xx on the raw PolyLib rows ----
 * One warp per problem, lane = input row (a row is converted by one lane exactly as the host does it);
 * an equality row also writes its negated copy, so the output row of a lane is its index plus the
 * equalities before it (ballot + popc).  lane 0 writes the descriptor. */
template <class T>
__global__ void __launch_bounds__(256) pip_convert_kernel(const PipConvertArgs A)
{
  const int lane = threadIdx.x & 31;
  const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
  const PipConvertShape &S = A.s;
  int max_nl = 0, max_nm = 0, nwide = 0;
  for (long long p = warp; p < A.n; p += nwarps) {
    T *tab = (T *)A.pool + p * A.stride;
    pip_i64 lost = 0;
    int nl = 0, nm = 0;
    for (int b0 = 0; b0 < S.dr; b0 += 32) {
      const int i = b0 + lane;
      const bool in = i < S.dr;
      const pip_i64 *row = A.dom + (p * S.dr + (in ? i : 0)) * (long long)S.dc;
      const bool eq = in && row[0] == 0;
      const unsigned eqm = __ballot_sync(0xffffffffu, eq), inm = __ballot_sync(0xffffffffu, in);
      if (in) {
        T *r = tab + (size_t)(nl + lane + __popc(eqm & ((1u << lane) - 1u))) * S.width;
        pip_convert_row<T>(row, S.dc, r, S.width, S.Nn, 0, S.Shift, S.Bg, S.Urs, lost);
        if (eq) pip_convert_negate<T>(r, r + S.width, S.width, lost);
      }
      nl += __popc(inm) + __popc(eqm);
    }
    if (S.has_ctx) {
      T *ctab = tab + (size_t)nl * S.width;
      for (int b0 = 0; b0 < S.cr; b0 += 32) {
        const int i = b0 + lane;
        const bool in = i < S.cr;
        const pip_i64 *row = A.ctx + (p * S.cr + (in ? i : 0)) * (long long)S.cc;
        const bool eq = in && row[0] == 0;
        const unsigned eqm = __ballot_sync(0xffffffffu, eq), inm = __ballot_sync(0xffffffffu, in);
        if (in) {
          T *r = ctab + (size_t)(nm + lane + __popc(eqm & ((1u << lane) - 1u))) * S.cwidth;
          pip_convert_row<T>(row, S.cc, r, S.cwidth, S.Np - S.Urs, 1, S.Shift, S.Bg - S.Nn - 1, S.Urs, lost);
          if (eq) pip_convert_negate<T>(r, r + S.cwidth, S.cwidth, lost);
        }
        nm += __popc(inm) + __popc(eqm);
      }
    }
    const bool wide = __any_sync(0xffffffffu, lost != 0);
    if (lane == 0) {
      PipProblem P;
      P.nvar = S.Nn; P.nparm = S.Np; P.ni = nl; P.nc = nm; P.bigparm = S.Bg;
      P.flags = S.pflags | (wide ? PIP_F_WIDE_INPUT : 0);
      P.off = p * A.stride;
      A.prob[p] = P;
    }
    max_nl = nl > max_nl ? nl : max_nl;
    max_nm = nm > max_nm ? nm : max_nm;
    nwide += wide ? 1 : 0;
  }
  if (lane == 0 && A.dims) {
    atomicMax(A.dims + 0, max_nl);
    atomicMax(A.dims + 1, max_nm);
    if (nwide) atomicAdd(A.dims + 2, nwide);
  }
}

extern "C" cudaError_t pip_launch_convert(const PipConvertArgs *A, int elem_log2, cudaStream_t stream)
{
  long long blocks = (A->n + 7) / 8;
  if (blocks > 148 * 16) blocks = 148 * 16;
  if (blocks < 1) blocks = 1;
  if (elem_log2 == 2) pip_convert_kernel<int><<<(int)blocks, 256, 0, stream>>>(*A);
  else pip_convert_kernel<pip_i64><<<(int)blocks, 256, 0, stream>>>(*A);
  return cudaGetLastError();
}

/* ---- caller arrays in device memory (pip_solve_dense_dp): a chunk's per-problem results, written where the
 * caller keeps them.  The same mapping the host applies to a staged chunk: a status that is not final becomes
 * PIP_ST_CAPACITY (and its report all zero), a span is the chunk's base plus the problem's slot offset, a length
 * loses its narrow flag. */
__global__ void __launch_bounds__(256) pip_emit_device_kernel(const int *st, const pip_u64 *hs, const long long *off,
                                                              const long long *len, const PipInfo *inf, long long n,
                                                              long long base, int *status, pip_u64 *hashes,
                                                              long long *ser_off, long long *ser_len, PipInfo *info)
{
  const long long i0 = (long long)blockIdx.x * blockDim.x + threadIdx.x, step = (long long)gridDim.x * blockDim.x;
  for (long long i = i0; i < n; i += step) {
    const int s0 = st[i];
    const bool final = PIP_STATUS_IS_FINAL(s0);
    status[i] = final ? s0 : PIP_ST_CAPACITY;
    if (hashes) hashes[i] = hs[i];
    if (ser_off) ser_off[i] = base + off[i];
    if (ser_len) ser_len[i] = len[i] & ~PIP_LEN_NARROW;
    if (info) {
      const PipInfo zero = {0, 0, 0, 0, 0, 0, {0, 0}};
      info[i] = final ? inf[i] : zero;
    }
  }
}
extern "C" cudaError_t pip_launch_emit_device(const int *st, const pip_u64 *hs, const long long *off, const long long *len,
                                              const PipInfo *inf, long long n, long long base, int *status, pip_u64 *hashes,
                                              long long *ser_off, long long *ser_len, PipInfo *info, cudaStream_t stream)
{
  long long blocks = (n + 255) / 256;
  if (blocks > 148 * 8) blocks = 148 * 8;
  if (blocks < 1) blocks = 1;
  pip_emit_device_kernel<<<(int)blocks, 256, 0, stream>>>(st, hs, off, len, inf, n, base, status, hashes, ser_off, ser_len,
                                                          info);
  return cudaGetLastError();
}

/* single-CTA exclusive scan of ncells (n up to a few million: 1024 threads, chunked) */
__global__ void pip_scan_kernel(const PipResult *res, const int *order, long long *dst_off, int nprob, long long *total,
                                int ser_mode)
{
  __shared__ long long warp_sums[32];
  __shared__ long long carry;
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  if (tid == 0) carry = 0;
  __syncthreads();
  for (int base = 0; base < nprob; base += blockDim.x) {
    const int i = base + tid;
    long long v = 0;
    if (i < nprob) {
      const PipResult &r = res[order ? order[i] : i];
      if (ser_mode) v = (r.rflags & PIP_RES_SER32) ? ((long long)r.ser_words + 1) / 2 : (long long)r.ser_words;
      else v = (long long)r.ncells * ((r.rflags & PIP_RES_WIDE) ? 3 : 1);
    }
    long long x = v;
    for (int o = 1; o < 32; o <<= 1) {
      long long y = __shfl_up_sync(0xffffffffu, x, o);
      if (lane >= o) x += y;
    }
    if (lane == 31) warp_sums[wid] = x;
    __syncthreads();
    if (wid == 0) {
      long long s = (lane < (int)(blockDim.x >> 5)) ? warp_sums[lane] : 0;
      for (int o = 1; o < 32; o <<= 1) {
        long long y = __shfl_up_sync(0xffffffffu, s, o);
        if (lane >= o) s += y;
      }
      warp_sums[lane] = s;
    }
    __syncthreads();
    const long long before = carry + (wid ? warp_sums[wid - 1] : 0) + (x - v);
    if (i < nprob) dst_off[i] = before;
    __syncthreads();
    if (tid == blockDim.x - 1) carry = before + v;
    __syncthreads();
  }
  if (tid == 0) *total = carry;
}

extern "C" cudaError_t pip_launch_gather(PipResult *res, const int *order, const PipCell *cells, long long *dst_off,
                                         pip_u64 *out, int nprob, long long *total, int phase,
                                         cudaStream_t stream)
{
  if (phase == 0 || phase == 2) pip_scan_kernel<<<1, 1024, 0, stream>>>(res, order, dst_off, nprob, total, phase == 2);
  else {
    int blocks = (nprob + 7) / 8;
    if (blocks > 148 * 16) blocks = 148 * 16;
    if (blocks < 1) blocks = 1;
    pip_gather_kernel<<<blocks, 256, 0, stream>>>(res, order, cells, dst_off, out, nprob);
  }
  return cudaGetLastError();
}
