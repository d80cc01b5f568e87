/* Shared host/device plain-data types of the batched PipLib solver core.
 *
 * Vocabulary follows the reference (paths relative to the reference tree):
 *   tableau row flags    source/tab.h:58-63
 *   solution cell kinds  source/sol.c:42-50, cell = {flags, param1, param2} source/sol.c:37-40
 *   hard limits          source/type.h:39,49,50 and source/tab.h:70
 */
#ifndef PIP_TYPES_H
#define PIP_TYPES_H

#include <stdint.h>

typedef long long pip_i64;
typedef unsigned long long pip_u64;

/* row flags */
enum { PIP_UNIT = 1, PIP_PLUS = 2, PIP_MINUS = 4, PIP_ZERO = 8, PIP_CRITIC = 16, PIP_UNKNOWN = 32 };
/* packed position word: flag | link << 8 (link = unit column or storage slot) */
#define PIP_FLAG(x) ((x) & 0xff)
#define PIP_LINK(x) ((x) >> 8)
#define PIP_MKFL(f, l) ((f) | ((l) << 8))
/* cell kinds */
enum { PIP_C_FREE = 0, PIP_C_NIL = 1, PIP_C_IF = 2, PIP_C_LIST = 3, PIP_C_FORM = 4, PIP_C_NEW = 5,
       PIP_C_DIV = 6, PIP_C_VAL = 7, PIP_C_ERROR = 8 };
/* problem flags (traiter flags, source/funcall.h:34-35, + our own) */
enum { PIP_F_INT = 1, PIP_F_DUAL = 2, PIP_F_DEEPEST = 4,
       PIP_F_SIMPLE_SER = 8,      /* cells -> quast words without column surgery: the solver sizes the stream itself */
       PIP_F_WIDE_INPUT = 16 };   /* device-side conversion: some input value left int32 (the int32 pool holds garbage
                                     for this problem; it is solved from the int64 pool built on demand) */

/* phases of the -DPIP_PROFILE cycle accounting */
enum { PIP_PH_LOAD = 0, PIP_PH_SORT, PIP_PH_SCAN, PIP_PH_BUILDSUB, PIP_PH_CHOOSE, PIP_PH_UPDATE, PIP_PH_SWAP,
       PIP_PH_CUT, PIP_PH_FRAME, PIP_PH_EMIT, PIP_PH_OTHER,
       PIP_PH_U_HEAD, PIP_PH_U_PASS1, PIP_PH_U_GCD, PIP_PH_U_DIV, PIP_PH_U_WAIT, PIP_NPHASE };

#define PIP_LEVEL_S_WIDE 100       /* slack level of the int32 shared-memory class when it has room (pip_slack) */
#define PIP_SOL_SIZE 4096
#define PIP_MAXCOL 512
#define PIP_MAXPARM 50
#define PIP_MAX_DET 4

/* per-problem status.  0/1 and 1000+exit-code are the reference's verdicts (see
 * include/piplib_b200.h); the 4xxx codes are internal scheduling states that never reach the
 * caller: the host re-runs such a problem in a larger size class. */
enum {
  PIP_ST_OK = 0,
  PIP_ST_VOID = 1,
  PIP_ST_FATAL = 1000,           /* + exit code of the reference */
  PIP_ST_FAULT = 2000,           /* division by zero: the reference dies of SIGFPE */
  PIP_ST_PENDING = 4000,         /* not solved yet (warp arena exhausted / not reached) */
  PIP_ST_CAPACITY = 4001,        /* exceeded the working-set capacity of its size class */
  PIP_ST_UNSUPPORTED = 4002,
  PIP_ST_WIDEN = 4003            /* int32 instantiation: needs the int64 kernel */
};

typedef struct {
  int nvar, nparm, ni, nc;       /* unknowns, parameters, tableau rows, context rows */
  int bigparm;                   /* tableau column of the big parameter or -1 */
  int flags;                     /* PIP_F_* */
  pip_i64 off;                   /* word offset into the input pool: ni*(nvar+nparm+1) tableau
                                    words (row-major, .dat column order) then nc*(nparm+1) */
} PipProblem;

typedef struct {
  int status;
  int ncells;
  pip_i64 cell_off;              /* first cell in the cell pool; after the gather: word offset
                                    into the compact stream */
  unsigned pivots;               /* successful pivots incl. sub-solves */
  unsigned cuts;
  unsigned subsolves;            /* non-parametric feasibility solves (compa_test, context) */
  unsigned splits;
  unsigned max_rows, max_cols;   /* largest nligne x ncol seen by a pivot */
  unsigned ser_words;            /* words of the serialised quast (device-side decode), else 0 */
  unsigned elem_updates_lo, elem_updates_hi;
  unsigned rflags;               /* PIP_RES_* */
} PipResult;

typedef struct {
  int kind;
  int pad;
  pip_i64 p1, p2;
} PipCell;

/* per-problem parameters of the cells -> quast decode (source/piplib.c:866-867: Bg-Nn-1, Urs_parms,
 * sol_flags) for the device-side serialiser */
typedef struct {
  int bg, urs, flags;
} PipDecodeParm;

/* Wire format of the solution cells after the device-side gather: one 64-bit word per cell,
 *   bits 0-3 kind | bits 4-19 param2 (unsigned, denominators) | bits 20-63 param1 (signed),
 * unless some cell of the problem does not fit (PIP_RES_WIDE in PipResult.rflags): then the
 * problem's cells are shipped as raw {kind, param1, param2} triples (3 words per cell). */
#define PIP_RES_WIDE 1u
#define PIP_RES_SER32 2u          /* device-decode mode: the quast words were shipped as int32 */
#define PIP_RES_SIZED 4u          /* ser_words was computed by the solver (PIP_F_SIMPLE_SER) */
#define PIP_RES_WORDS 16u         /* word mode: the window holds the serialised quast words, not cells */
#define PIP_RES_SRC32 32u         /* word mode: those words are int32 (class S32), else int64 */
#define PIP_RES_WRAPPED 8u        /* int64 classes: an exact 128-bit product of a pivot update left 64 bits (the
                                     reference wraps silently there; its own verdict is reported unchanged) */
#define PIP_CELL_FITS(p1, p2) ((pip_u64)(p2) < 65536ull && (p1) >= -(1ll << 43) && (p1) < (1ll << 43))
#define PIP_CELL_PACK(kind, p1, p2) ((pip_u64)(unsigned)(kind) | ((pip_u64)(p2) << 4) | ((pip_u64)(p1) << 20))
#define PIP_CELL_KIND(w) ((int)((w) & 15ull))
#define PIP_CELL_P2(w) ((pip_i64)(((w) >> 4) & 0xffffull))
#define PIP_CELL_P1(w) (((pip_i64)(w)) >> 20)

/* Device-side decode with span reservation (dense path): the decoding warp reserves the problem's span of
 * the compact word buffer with one atomic add, so neither a scan kernel nor a host round trip sits between
 * the solve and the decode; per-problem results land in structure-of-arrays form (no 56-byte records cross
 * PCIe), counters are summed on the device. */
typedef struct {
  unsigned long long *ctl;       /* [0] 64-bit slots reserved so far, [1] problems with a final status (this
                                    launch), [2] set when a span did not fit `cap`, [3] spare */
  long long cap;                 /* 64-bit slots in the compact buffer */
  int words64;                   /* 1: every word is written as int64; 0: int32 words for PIP_RES_SER32 problems */
  int *status;
  pip_u64 *hash;
  long long *off;                /* slot offset of the problem's span in the compact buffer */
  long long *len;                /* words; bit 62 set when they were written as int32 */
  unsigned long long *stats;     /* [PIP_SO_NSTAT]: pivots, cuts, subsolves, splits, elem_updates, cells, max_rows,
                                    max_cols, problems flagged PIP_RES_WRAPPED (final statuses only) */
  struct PipInfo *info;          /* per-problem report (PipProblemInfo_dp) or NULL when the caller did not ask for it */
} PipStreamOut;

/* the per-problem report of the dense path, PipProblemInfo_dp of include/piplib_b200.h: the counters of the
 * record a verdict came with; all zero for a status that is no verdict of the reference (4xxx) */
typedef struct PipInfo {
  unsigned flags, pivots, cuts, splits, max_rows, max_cols, spare[2];
} PipInfo;
#define PIP_INFO_FLAG_WRAPPED 1u         /* = PIP_FLAG_WRAPPED */
#define PIP_LEN_NARROW (1ll << 62)
#define PIP_SO_NSTAT 9
enum { PIP_SO_SLOTS = 0, PIP_SO_FINALS = 1, PIP_SO_OVERFLOW = 2, PIP_SO_NCTL = 4 };
#define PIP_STATUS_IS_FINAL(st) ((st) != PIP_ST_PENDING && (st) != PIP_ST_CAPACITY && (st) != PIP_ST_WIDEN)

/* the working arena of one problem, carved by pip_layout (pip_solver.h); word offsets into the arena */
typedef struct PipTab {          /* warp-uniform, lives in registers */
  int den, fl, data, det;   /* word offsets into the arena */
  int stride, pcap, rcap;   /* words per slot, position capacity, slot capacity */
  int nvar, nparm, ni;
  int ldet;
} PipTab;

typedef struct PipLayout {
  PipTab m, s;
  int ctx, cstride, crcap;
  int cut, tmp;
  int total;
} PipLayout;

/* ---- subtree donation (SURVEY.md 8e: independent subtrees of one problem's parametric tree) ----------------
 * At a split the ELSE continuation is a self-contained work item: a snapshot of the tableau and the context
 * in the warp's frame stack (source/traiter.c:717,741-758: THEN runs on a copy, ELSE continues in the frame).
 * A warp that sees idle warps OFFERS the bottom frame of its stack -- the ELSE branch of its outermost open
 * split; everything the donor still does precedes that subtree in pre-order.  An idle warp CLAIMS the offer
 * (compare-and-swap on its state), restores the frame from the donor's stack, solves the subtree into its own
 * window as a new SEGMENT of the problem's stream and links the segment right after the donor's (so later,
 * inner donations of the same donor come before earlier, outer ones: pre-order).  An offer nobody claimed is
 * reclaimed by its owner when it gets there.  The copy kernel walks the segment list: first fatal verdict in
 * pre-order wins, the exit(26) cell limit is resolved from per-segment high-water marks, CAPACITY / WIDEN in
 * any segment re-runs the whole problem one class up. */
typedef struct {
  int problem;                   /* index into prob / res */
  int parent_seg;                /* the donor's segment: -1 = the problem's own (head) segment, else an offer index */
  int state;                     /* PIP_OFFER_* */
  int pad;
  const pip_i64 *frame;          /* the ELSE continuation in the donor's frame stack */
} PipOffer;
enum { PIP_OFFER_NONE = 0, PIP_OFFER_OPEN = 1, PIP_OFFER_CLAIMED = 2, PIP_OFFER_RECLAIMED = 3,
       PIP_OFFER_COPIED = 4 };      /* the thief has the frame in its own arena: the donor may reuse its stack */
enum { PIP_STL_OFFERS = 0, PIP_STL_IDLE = 1, PIP_STL_TOTAL = 2, PIP_STL_CURSOR = 3, PIP_STL_CLAIMS = 4, PIP_STL_NCTL = 8 };
typedef struct {
  int mode;                      /* 0 off; 1 on; 2 test: every offer is taken by its owner once it finished
                                    its own problem (exercises the whole splice on one warp, emulator) */
  int cap;                       /* offers = segments (a claimed offer becomes the segment of the same index) */
  PipOffer *offers;
  unsigned *ctl;                 /* [PIP_STL_*]: offers published, idle warps, warps of the launch, test cursor */
  PipResult *segs;               /* record of segment i (as PipResult: status, ncells, cell_off, counters, ser_words) */
  int *seg_next;                 /* segment after segment i in pre-order, -1 = none */
  int *seg_hwm;                  /* largest cell count segment i checked against SOL_SIZE (source/sol.c:96-100) */
  int *head_next;                /* per problem: first donated segment after the head segment, -1 = none */
  int *head_hwm;                 /* per problem: the head segment's high-water mark */
} PipSteal;

/* launch parameters of the warp-per-problem kernels */
typedef struct {
  const PipProblem *prob;
  const void *pool;              /* input words, 1 << pool_elem_log2 bytes each (int8/int32/int64) */
  int pool_elem_log2;
  const int *order;              /* optional permutation of problem indices (may be NULL) */
  int nprob;
  PipResult *res;
  PipCell *cells;                /* cell pool, cells_per_warp per warp */
  pip_i64 cells_per_warp;
  pip_i64 *stack;                /* split-frame stack pool (global memory) */
  pip_i64 stack_words_per_warp;
  pip_i64 *gwork;                /* working arenas in global memory (class G) or NULL (class S) */
  int work_words;                /* words of working arena per warp */
  unsigned *queue;               /* [0] next problem, [2] problems handed over (budget), [3] next entry of heavy[] */
  int sol_size, maxcol, maxparm;
  int slack_level;
  unsigned long long *prof;      /* [PIP_NPHASE] cycle sums (profile build only) or NULL */
  int have_layout;               /* every problem of the launch has the shape `layout` was carved for (dense batches):
                                    the arena layout comes from the host, pip_layout does not run per problem */
  PipLayout layout;
  const pip_i64 *images;         /* arena images of the problems (pip_image_kernel), indexed like prob, or NULL */
  int image_words, image_w1;     /* words per image; words of its first region (tableau), the context follows */
  PipSteal steal;                /* subtree donation (word mode only) */
  int emit_words;                /* word mode: PIP_F_SIMPLE_SER problems write their serialised quast (pip_solver.h) */
  /* ---- heavy-problem hand-over: the tail of a big launch is a few problems with very large parametric trees
   * (loop nests: mean 66 pivots, 1 in 10^4 above 2000), each on one warp while the machine idles.  A problem
   * that reaches a split with more than `budget` pivots behind it stops, is listed in heavy[] and keeps its
   * PENDING record; a second launch (from_heavy) of the instantiation with subtree donation solves the list
   * from scratch with every warp cooperating. */
  unsigned budget;               /* 0 = no hand-over */
  unsigned heavy_max;            /* no more hand-overs once this many are listed (a batch of heavy problems only is
                                    balanced by problems; a few more may slip in: the count is read, not reserved) */
  int *heavy;                    /* [nprob] problems handed over, queue[2] of them */
  int from_heavy;                /* this launch solves heavy[0 .. queue[2]) (cursor queue[3]) instead of order[0 .. nprob) */
  int heavy_warps;               /* ... with at most this many warps per listed problem (the others leave at once) */
  pip_i64 heavy_region;          /* ... and the cells of the launch's whole region (shared out among the warps that stay) */
  pip_i64 cell_base;             /* first cell of this launch's windows in `cells` (the second launch writes behind the first) */
} PipLaunch;

#endif
