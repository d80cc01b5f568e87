/* piplib-b200: the batched C-ABI (new; not in the reference) + status vocabulary.
 *
 * Everything here is plain C: pointers, sizes, ints.  No CUDA or torch types cross the boundary.
 *
 * Entry points and the reference interface each one replaces or extends:
 *
 *   pip_solve_batch_dp        n independent pip_solve_dp calls (source/piplib.c:722-880) in one
 *                             device batch; out[i] is the same tree pip_solve_dp would return.
 *   pip_traiter_batch_dp      n independent runs of the CLI's per-problem body
 *                             (source/maind.c:150-232: tab_get x2, tab_simplify, context check,
 *                             traiter_xx) on already-lexed tableaus; returns raw solution cells
 *                             ({flags, param1, param2}, source/sol.c:37-40).
 *   pip_solve_dense_dp        pip_solve_batch_dp for a batch whose problems share one shape,
 *                             given as two dense int64 arrays (no PipMatrix objects); returns
 *                             cells or a hash per problem.  This is the bulk path used by
 *                             bench.py (host buffers in, host buffers out); it also reads and
 *                             writes caller arrays in device memory.
 *   pip_solve_dense_info_dp   pip_solve_dense_dp plus a per-problem report: the int64 overflow flag and the
 *                             pivot, cut and split counts (PipProblemInfo_dp).
 *   pip_device_*              the same batch with inputs/outputs resident in device memory
 *                             (kernel-only timing; pointers are CUdeviceptr values as integers).
 *   pip_quast_serialize_dp    PipQuast -> int64 stream (test/interop helper).
 *
 * Status codes (per problem):
 *   0       solved
 *   1       the context is empty: pip_solve_dp returns NULL, the CLI prints "void"
 *   1000+c  the reference prints a message and calls exit(c) (source/traiter.c:424-427,441-444:
 *           "Integer overflow" c=1; source/traiter.c:174-177,710-713: "Too much parameters"
 *           c=1/2; source/integrer.c:324-327: "Too many variables" c=3; source/sol.c:97-100:
 *           "The solution is too complex! : sol" c=26; assert(ok_var) integrer.c:499: c=134)
 *   2000    the reference dies of a division by zero (SIGFPE) after a silent int64 wrap
 *   4001    problem exceeds the largest device size class (never seen on the fixtures)
 *   4002    option not implemented on the device (Compute_dual, Deepest_cut)
 * pip_solve_dp (batch of one) keeps the reference behaviour: message on stderr + exit(c).
 */
#ifndef PIPLIB_B200_H
#define PIPLIB_B200_H

#include <stddef.h>

#include <piplib/piplib.h>

#if defined(__cplusplus)
extern "C" {
#endif

#define PIP_STATUS_OK 0
#define PIP_STATUS_VOID 1
#define PIP_STATUS_FATAL 1000
#define PIP_STATUS_FAULT 2000
#define PIP_STATUS_TOO_LARGE 4001
#define PIP_STATUS_UNSUPPORTED 4002

typedef struct {
  int kind;                 /* Free0 Nil1 If2 List3 Form4 New5 Div6 Val7 (source/sol.c:42-50) */
  int pad;
  long long p1, p2;
} PipCell_dp;

typedef struct {
  int nvar, nparm, ni, nc;  /* .dat header fields Nn Np Nl Nm (doc/piplib.texi:570-586) */
  int bigparm;              /* Bg: tableau column of the big parameter, or -1 */
  int nq;                   /* bit 0: 1 integer, 0 rational (the .dat field); bit 1: rational with dual
                               variables (TRAITER_DUAL, no parameters); bit 2: deepest cuts (pip -d) */
} PipTableauHeader_dp;

typedef struct {
  unsigned long long pivots, cuts, subsolves, splits, elem_updates;
  unsigned max_rows, max_cols;
  double seconds_h2d, seconds_kernel, seconds_d2h, seconds_host;
  float device_ms;          /* CUDA-event time from the first to the last kernel of the batch */
  int launches;             /* kernels launched by the last batch call */
  int rounds;               /* solve launches (size-class escalations included) */
  unsigned long long h2d_bytes, d2h_bytes;
  unsigned long long cells;  /* solution cells produced by the batch */
  unsigned long long phase_cycles[16]; /* per-phase warp cycles, profile build only (else 0) */
  unsigned long long wrapped; /* problems in which an exact 128-bit product of a pivot update left int64: the
                                 reference wraps silently there (source/traiter.c:483-485) and so do we -- the answer is
                                 bit-identical -- but from that point on its verdict is "Integer overflow" or garbage
                                 (SURVEY.md section 8, P3).  Per problem: pip_last_batch_flags_dp. */
} PipBatchStats_dp;

/* n x pip_solve_dp.  options may be NULL (defaults) ; contexts[i] may be NULL (no parameters).
 * out[i] receives the tree (NULL when status[i] != 0); returns 0 or a negative CUDA/system error. */
int pip_solve_batch_dp(int n, PipMatrix_dp *const *domains, PipMatrix_dp *const *contexts,
                       const int *bignums, const PipOptions_dp *options,
                       PipQuast_dp **out, int *status);

/* n x (maind.c per-problem body).  tab[i]: ni x (nvar+nparm+1) row-major, .dat column order
 * [unknowns | constant | parameters]; ctx[i]: nc x (nparm+1).  cells_out must hold cell_cap cells;
 * cell_off[i]/ncells[i] locate problem i's cells.  Returns 0, -2 if cell_cap is too small (then
 * *cells_needed says how many), or a negative error. */
int pip_traiter_batch_dp(int n, const PipTableauHeader_dp *hdr, const long long *const *tab,
                         const long long *const *ctx, int *status, PipCell_dp *cells_out,
                         long long cell_cap, long long *cell_off, int *ncells, long long *cells_needed);

/* sol_simplify_xx (source/sol.c:272-288; `pip -z`) on one problem's cells as returned by
 * pip_traiter_batch_dp: cells may turn Free (kind 0) and *ncells may shrink.  Host only. */
void pip_cells_simplify_dp(PipCell_dp *cells, int *ncells);

/* make `cells` the solution space sol_quast_edit_dp (piplib.h) decodes from on this thread: the pair
 * replaces the reference's sol_init/traiter/sol_quast_edit sequence (source/piplib.c:853-867) for a
 * caller that drives the tableau-level entry point itself.  The cells are copied. */
void pip_cells_bind_dp(const PipCell_dp *cells, int ncells);

/* Dense batch through the pip_solve_dp path: dom is [n][dom_rows][dom_cols] (PolyLib rows),
 * ctx is [n][ctx_rows][ctx_cols] or NULL (has_ctx=0):
 *   status[i]  as above
 *   hashes[i]  (optional) hash of the serialised quast words (pip_hash_word: a sum of mixed (word, index) pairs; the function tests/ and
 *              oracle/ apply to the reference's trees); 0 when status[i] is fatal
 *   ser        (optional) the serialised quasts: problem i occupies
 *              ser[ser_off[i] .. ser_off[i] + ser_len[i]); spans are packed without gaps but, as
 *              chunks of the batch finish in any order, not in problem order.  ser_off has n+1
 *              entries, ser_off[n] = words used/needed; returns -2 when ser_cap is too small.
 * Returns 0, -2 (above), -3 (device buffers refused, below) or -1 (a CUDA or system error).
 *
 * Buffers may be host memory (pageable or page-locked, see pip_pin_buffer_dp) or device memory (cudaMalloc,
 * torch CUDA tensors; managed memory counts as host memory).  The inputs (dom and ctx) and the outputs
 * (status, hashes, ser, ser_off, ser_len: the non-NULL ones) are placed independently:
 *   device inputs   the rows are converted where they are; they never cross PCIe
 *   device outputs  every output, ser_off[n] included, is written in device memory, by the device
 * Device-resident buffers run on the device that owns them, whatever pip_set_device_dp / pip_set_devices_dp
 * say.  The call returns -3, before anything is written, when the device-resident arrays are on different
 * devices, when only one of dom / ctx is device-resident or only some of the outputs are, or when
 * device-resident buffers meet an option the host decoder serves (Simplify; Compute_dual with Nq = 0).
 * Ordering: the work that writes device inputs (or last used device outputs) must be complete when the call
 * is made -- the library runs on CUDA streams of its own -- and device outputs are complete when it returns.
 * The call is host-synchronous in every case. */
int pip_solve_dense_dp(long long n, int dom_rows, int dom_cols, const long long *dom,
                       int has_ctx, int ctx_rows, int ctx_cols, const long long *ctx,
                       int bignum, const PipOptions_dp *options,
                       int *status, unsigned long long *hashes,
                       long long *ser, long long ser_cap, long long *ser_off, long long *ser_len);

/* Per-problem solve report of a dense batch.  Each field equals, problem for problem, the field of the
 * oracle's per-problem statistics (oracle/pyoracle.py PortStats, oracle/pip_oracle.c) named beside it: */
typedef struct {
  unsigned flags;           /* wrapped > 0: PIP_FLAG_WRAPPED (bit 0), as pip_last_batch_flags_dp reports it: an exact
                               128-bit product of a pivot update left int64 (see PipBatchStats_dp.wrapped).  The
                               whole-grid class (non-parametric problems that outgrow the team classes) does not
                               detect the wrap: a problem it solves reports 0, there and in PipBatchStats_dp.wrapped */
  unsigned pivots;          /* pivots: successful pivots, those of compa_test / context feasibility sub-solves included */
  unsigned cuts;            /* cuts_const + cuts_parm: Gomory cuts, constant and parametric */
  unsigned splits;          /* splits: parametric splits (If nodes emitted by the main solve) */
  unsigned max_rows;        /* max_rows: the largest nligne (unknowns + rows) of a pivot */
  unsigned max_cols;        /* max_cols: the largest ncol of a pivot */
  unsigned spare[2];        /* zero */
} PipProblemInfo_dp;        /* 32 bytes */

/* pip_solve_dense_dp, and the report of problem i in info[i] (NULL: none; pip_solve_dense_dp is this call with
 * info = NULL).  info is an output like status / hashes / ser: host or device memory, placed with the other
 * outputs (a device-resident info beside host outputs, or the reverse, returns -3 before anything is written).
 * The record belongs to the attempt that gave the final status: a problem re-run one size class up, handed over
 * to the cooperative launch or to the whole-grid class reports that last run only; under subtree donation it is
 * the sum over the problem's segments up to the verdict.  For a fatal status (1000+c, 2000) the counters are those
 * at the verdict (a cell-limit verdict, 1026, met inside a donated subtree cannot be placed in it: such a problem
 * is solved once more without donation); for 4001 / 4002 the record is all zero.  Same return codes as
 * pip_solve_dense_dp. */
int pip_solve_dense_info_dp(long long n, int dom_rows, int dom_cols, const long long *dom,
                            int has_ctx, int ctx_rows, int ctx_cols, const long long *ctx,
                            int bignum, const PipOptions_dp *options,
                            int *status, unsigned long long *hashes,
                            long long *ser, long long ser_cap, long long *ser_off, long long *ser_len,
                            PipProblemInfo_dp *info);

/* Page-lock a caller buffer (cudaHostRegister, visible to every device) so that pip_solve_dense_dp moves
 * it by DMA alone: input arrays `dom` / `ctx` registered this way are uploaded as they are and converted to
 * tableaus on the device (tab_Matrix2Tableau_xx, source/tab.c:292-393, as a kernel); an output stream
 * `ser` registered this way receives the serialised quasts straight from the device.  Buffers allocated
 * page-locked by the caller (cudaHostAlloc, torch pin_memory) are recognised without this call.  Pageable
 * buffers keep working: they are converted / widened by the host thread pool through pinned staging.
 * The answers are identical either way.  Returns 0 or -1. */
int pip_pin_buffer_dp(void *p, size_t bytes);
int pip_unpin_buffer_dp(void *p);
/* page-locked memory allocated by the driver (cudaHostAlloc, portable): the fastest DMA source / target;
 * registering existing memory (above) pins 4 KB pages in place and transfers a little slower */
void *pip_alloc_pinned_dp(size_t bytes);
void pip_free_pinned_dp(void *p);

/* Devices pip_solve_dense_dp spreads a batch over (one process, several GPUs): the chunks of a batch go
 * to whichever device has a free lane (a shared queue: dynamic balance across the GPUs), results land in
 * the caller's arrays as for one device.  n = 0 returns to the single default device (pip_set_device_dp). */
int pip_set_devices_dp(int n, const int *devices);

/* Device-resident variant of the dense batch: converted and uploaded once by create(); run()
 * executes only kernels: with fetch_cells = 0 the whole device job (solve + decode to serialised quasts,
 * statuses and hashes, all left in HBM; nothing per problem crosses PCIe unless a problem has to change
 * size class), with fetch_cells = 1 solve + cell gather and the cells copied to the host.  A job of more
 * than 2^19 problems is run in three parts on engine lanes of their own (the tail of a part -- its few
 * largest trees -- is filled by the next part); device_ms is then the time from the first launch to the
 * end of the last part. */
typedef struct pip_device_batch pip_device_batch;
pip_device_batch *pip_device_batch_create(long long n, int dom_rows, int dom_cols, const long long *dom,
                                          int has_ctx, int ctx_rows, int ctx_cols, const long long *ctx,
                                          int bignum, const PipOptions_dp *options);
int pip_device_batch_run(pip_device_batch *b, int fetch_cells, float *device_ms);
/* results of the last run: status always; hashes if that run decoded on the device (fetch_cells = 0) or fetched the cells.
 * They are read out of the engines' buffers in HBM: call it before the next solve on the same device. */
int pip_device_batch_results(pip_device_batch *b, int *status, unsigned long long *hashes);
/* the per-problem reports of the last run (PipProblemInfo_dp, n records) into a host array; read like the results.
 * A run that decodes on the device (fetch_cells = 0) writes them only when they were asked for: info = NULL makes
 * every later run of b write them (returns 0); the reports of a run that did not write them return -3. */
int pip_device_batch_info(pip_device_batch *b, PipProblemInfo_dp *info);
void pip_device_batch_destroy(pip_device_batch *b);

/* One LARGE non-parametric tableau solved by the whole grid (BASELINE config 4; the tableau lives
 * in HBM, the pivot update is HBM-bound).  tab is ni x (nvar+1), .dat column order; nq as in the
 * .dat header; cut_rows = spare rows for Gomory cuts; sol_size / maxcol = 0 keep the reference's
 * limits (source/type.h:39,49: a 4096-unknown solution needs 8193 cells, so the stock limits end
 * in status 1026 exactly like the reference).  Same semantics as the maind.c per-problem body. */
typedef struct pip_large_problem pip_large_problem;
pip_large_problem *pip_large_create_dp(int nvar, int ni, int nq, const long long *tab, int cut_rows,
                                       int sol_size, int maxcol);
int pip_large_run_dp(pip_large_problem *p, float *kernel_ms);
int pip_large_fetch_dp(pip_large_problem *p, int *status, PipCell_dp *cells, int cell_cap, int *ncells,
                       long long *info /* [12]: pivots, cuts, skipped identity rows, final ni,
                                          SM cycles in the row/column-choice phase, in the update phase,
                                          then sub-phases: swap, row pick, column choice, determinant,
                                          active-row list, spare */);
void pip_large_destroy_dp(pip_large_problem *p);

void pip_last_batch_stats_dp(PipBatchStats_dp *out);
/* per-problem flags of the last pip_solve_batch_dp / pip_traiter_batch_dp call on this thread
 * (bit 0 = PIP_FLAG_WRAPPED, see PipBatchStats_dp.wrapped); returns the number of problems of that call */
#define PIP_FLAG_WRAPPED 1u
long long pip_last_batch_flags_dp(unsigned *flags, long long cap);

/* PipQuast -> int64 stream; returns the number of words (may exceed cap: nothing past cap is written) */
long pip_quast_serialize_dp(const PipQuast_dp *q, long long *out, long cap);

int pip_set_device_dp(int device);                     /* select the CUDA device (default 0) */
/* Subtree donation inside one problem's parametric tree (dense path, bulk batches): idle warps take over the
 * ELSE branches other warps offer (source/traiter.c:717,741-758: the THEN branch runs on a copy, the ELSE branch
 * is a self-contained continuation) and the segments are spliced in pre-order -- same quasts, same verdicts.
 * mode < 0: automatic (small batches of parametric problems, where most warps would idle), 0: off, > 0: on. */
void pip_set_donation_dp(int mode);
const char *pip_b200_version(void);

#if defined(__cplusplus)
}
#endif
#endif
