/* Subtree donation, result side (PipSteal in pip_types.h): a problem whose subtrees were solved by other warps
 * is a list of SEGMENTS in pre-order -- the head segment (the problem's own record) and the donated ones.
 * This walk decides the problem's verdict exactly as the sequential reference would have met it:
 *   - the first segment in pre-order that did not finish OK gives the status (a fatal verdict of the
 *     reference, or CAPACITY / WIDEN: the whole problem is re-run one class up);
 *   - the cell limit of sol_alloc (source/sol.c:96-100) is checked with the cells of all earlier segments as
 *     the base of each segment's high-water mark;
 * and sums what the segments counted up to the verdict: the head and every segment before the one that gave the
 * verdict, and that segment itself, whose counters stop at its verdict -- what the sequential reference counted
 * when it met it.  One verdict cannot be placed this way: the cell limit met inside a donated segment (the
 * segment does not know how many cells precede it, so it ran past the point where the reference stopped);
 * `verdict_seg` tells it apart.  Shared by the copy kernel and the emulator driver. */
#ifndef PIP_SEGMENTS_H
#define PIP_SEGMENTS_H

#include "pip_types.h"
#include "simt.h"

typedef struct {
  int status;
  int nseg;                      /* segments, the head included */
  int verdict_seg;               /* the donated segment that gave a status other than OK, -1 = none (or the head) */
  long long words, cells;
  unsigned long long pivots, cuts, subsolves, splits, elem_updates;
  unsigned max_rows, max_cols;
  unsigned all_flags_and, any_flags_or;      /* over the segments' rflags */
} PipResolved;

PIP_HD void pip_resolve_add(PipResolved &o, const PipResult &r)
{
  o.nseg++;
  o.words += r.ser_words; o.cells += r.ncells;
  o.pivots += r.pivots; o.cuts += r.cuts; o.subsolves += r.subsolves; o.splits += r.splits;
  o.elem_updates += ((unsigned long long)r.elem_updates_hi << 32) | r.elem_updates_lo;
  o.max_rows = r.max_rows > o.max_rows ? r.max_rows : o.max_rows;
  o.max_cols = r.max_cols > o.max_cols ? r.max_cols : o.max_cols;
  o.all_flags_and &= r.rflags; o.any_flags_or |= r.rflags;
}

PIP_HD void pip_resolve_segments(const PipResult &head, int head_next, const PipSteal &S, int sol_size, PipResolved &o)
{
  o.status = head.status; o.nseg = 0; o.verdict_seg = -1; o.words = 0; o.cells = 0;
  o.pivots = o.cuts = o.subsolves = o.splits = o.elem_updates = 0;
  o.max_rows = o.max_cols = 0; o.all_flags_and = 0xffffffffu; o.any_flags_or = 0;
  pip_resolve_add(o, head);
  if (head.status != PIP_ST_OK) return;                  /* the head's verdict comes first in pre-order */
  for (int s = head_next; s >= 0; s = S.seg_next[s]) {
    const PipResult r = S.segs[s];
    if (r.status != PIP_ST_OK) { o.status = r.status; o.verdict_seg = s; pip_resolve_add(o, r); return; }
    if (o.cells + (long long)S.seg_hwm[s] >= (long long)sol_size) {
      o.status = PIP_ST_FATAL + 26; o.verdict_seg = s; pip_resolve_add(o, r); return;
    }
    pip_resolve_add(o, r);
  }
}

/* the per-problem report (PipInfo) of a record, resolved over its segments or not */
PIP_HD PipInfo pip_info_of(const PipResult &r)
{
  PipInfo o = {0, 0, 0, 0, 0, 0, {0, 0}};
  if (r.status >= PIP_ST_PENDING) return o;
  o.flags = (r.rflags & PIP_RES_WRAPPED) ? PIP_INFO_FLAG_WRAPPED : 0u;
  o.pivots = r.pivots; o.cuts = r.cuts; o.splits = r.splits;
  o.max_rows = r.max_rows; o.max_cols = r.max_cols;
  return o;
}

#endif
