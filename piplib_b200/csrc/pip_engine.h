/* Host-side batch engine: owns the device buffers, drives the size-class ladder
 * (S: shared-memory arenas, G3..G8: global-memory arenas of growing capacity), compacts and
 * fetches the solution cells.  Internal to the library (the C-ABI is include/piplib_b200.h). */
#ifndef PIP_ENGINE_H
#define PIP_ENGINE_H

#include <cuda_runtime.h>

#include <vector>

#include "pip_types.h"

struct PipBatchIn {
  size_t n = 0;
  const PipProblem *h_prob = nullptr;   /* host descriptors: always required (class planning) */
  const void *h_pool = nullptr;         /* host pool, uploaded unless d_pool is given */
  size_t pool_words = 0;                /* elements in the pool */
  int elem_log2 = 3;                    /* log2(bytes per pool element): 0, 2 or 3 */
  const PipProblem *d_prob = nullptr;   /* optional device-resident copies */
  const void *d_pool = nullptr;
  bool fetch_cells = true;              /* copy the compacted cells back to the host */
  const PipDecodeParm *h_decode = nullptr; /* if set: decode on the device, ship serialised quast words
                                              (+ hashes) instead of cells */
  int sol_size = PIP_SOL_SIZE, maxcol = PIP_MAXCOL;
  /* ---- dense path (pip_solve_dense_dp) ---- */
  const PipProblem *uniform = nullptr;  /* every problem has this shape (ni / nc = the maxima over the batch): the
                                           plan is made once, h_prob may be NULL when d_prob is given */
  const PipDecodeParm *uniform_decode = nullptr;   /* device decode, one parameter set for every problem */
  bool stream_out = false;              /* decode with span reservation; the serialised words and the per-problem
                                           arrays stay on the device (PipBatchOut::dev), nothing per problem
                                           crosses PCIe inside run() unless a problem has to change class */
  bool words64 = false;                 /* stream_out: every word as int64 (else int32 where it fits) */
  bool want_info = false;               /* stream_out: write the per-problem reports (PipDeviceOut::info) */
  bool overlapped = false;              /* other engine lanes run beside this batch: its tail is not idle time (no hand-over) */
  long long words_hint = 0;             /* stream_out: expected 64-bit slots for the whole batch (0 = default) */
  /* called when a problem's input does not fit the int32 pool (PIP_F_WIDE_INPUT): returns the int64 pool */
  const void *(*widen_pool)(void *ctx, cudaStream_t s) = nullptr;
  void *widen_ctx = nullptr;
};

/* device-resident results of a stream_out run: valid until the next run() on the same engine */
struct PipDeviceOut {
  const pip_i64 *words = nullptr;       /* compact buffer, 64-bit slots */
  long long slots = 0;                  /* slots used */
  const int *status = nullptr;
  const pip_u64 *hash = nullptr;
  const long long *off = nullptr, *len = nullptr;   /* per problem: slot offset, words | PIP_LEN_NARROW */
  const PipInfo *info = nullptr;        /* per problem: the report (PipBatchIn::want_info), else NULL */
  unsigned long long stats[PIP_SO_NSTAT] = {0};   /* pivots, cuts, subsolves, splits, elem_updates, cells, max_rows, max_cols, wrapped */
};

struct PipBatchTimes {
  double h2d = 0, kernel = 0, d2h = 0, total = 0;   /* seconds, wall clock around synchronised phases */
  float device_ms = 0;                               /* CUDA-event time first launch -> last kernel */
  int launches = 0, rounds = 0;
  size_t h2d_bytes = 0, d2h_bytes = 0;
  unsigned long long phase_cycles[PIP_NPHASE] = {0};   /* profile build only */
  float round_s[8] = {0};                              /* wall seconds of each solve round */
  int round_n[8] = {0};                                /* problems in each round */
};

/* read-only view of one problem's cells in the wire format (pip_types.h) */
struct PipCellView {
  const pip_u64 *w;
  bool wide;
  int n;
  int kind(int i) const { return wide ? (int)(w[3 * i] & 0xffffffffull) : PIP_CELL_KIND(w[i]); }
  pip_i64 p1(int i) const { return wide ? (pip_i64)w[3 * i + 1] : PIP_CELL_P1(w[i]); }
  pip_i64 p2(int i) const { return wide ? (pip_i64)w[3 * i + 2] : PIP_CELL_P2(w[i]); }
};

struct PipBatchOut {
  std::vector<PipResult> res;           /* cell_off = word offset into the round's host chunk */
  std::vector<const pip_u64 *> base;    /* per problem: base pointer of its round's host chunk */
  std::vector<pip_u64> hashes;          /* device-decode mode: hash of each serialised quast */
  PipBatchTimes times;
  PipDeviceOut dev;                     /* stream_out mode */
  PipCellView cells_of(size_t i) const
  {
    PipCellView v;
    v.w = base[i] ? base[i] + res[i].cell_off : nullptr;
    v.wide = (res[i].rflags & PIP_RES_WIDE) != 0;
    v.n = res[i].ncells;
    return v;
  }
};

class PipEngine {
 public:
  static PipEngine &get() { return lane(0); }
  /* independent engines (own stream + buffers) so that batches can be pipelined: while one lane
   * waits for its kernels, another converts inputs or decodes results; one set of lanes per device */
  enum { MAX_LANES = 8, MAX_DEVICES = 16 };
  static PipEngine &lane(int i);                 /* on the default device (pip_set_device_dp) */
  static PipEngine &at(int device, int lane);
  /* engine-owned device scratch for the caller's raw input rows and converted pool (dense path) */
  void *device_scratch(int which, size_t bytes);
  void *pinned_scratch(int which, size_t bytes);
  int device_id();
  /* engine-owned pinned staging for the input pool (valid until the next call on this lane) */
  void *pinned_input(size_t bytes);
  /* Runs the whole ladder.  Host cell storage referenced by `out` is engine-owned pinned memory,
   * valid until the next run() call.  Throws std::runtime_error on CUDA errors. */
  void run(const PipBatchIn &in, PipBatchOut &out);
  int set_device(int dev);
  int sm_count();
  cudaStream_t stream();
  struct Impl;

 private:
  PipEngine();
  Impl *impl_;
};

void pip_cuda_check(cudaError_t e, const char *what);
int pip_engine_device();
void pip_engine_set_donation(int mode);

#endif
