/* The C-ABI of piplib-b200 (include/piplib/piplib.h, include/piplib_b200.h).
 *
 * Host side of the boundary only: PolyLib matrix -> tableau conversion, option rewriting,
 * cell stream -> PipQuast decoding, printers, allocation.  All solving happens on the GPU
 * (pip_engine.cpp + pip_kernels.cu); there is no CPU solver in this library.
 *
 * Reference behaviour restated here (paths relative to the reference tree):
 *   pip_solve_xx            source/piplib.c:722-880
 *   tab_Matrix2Tableau_xx   source/tab.c:292-393
 *   sol_quast_edit_xx & co  source/sol.c:435-734   sol_simplify_xx source/sol.c:236-288
 *   printers / alloc / free source/piplib.c:176-619
 */
#include <ctype.h>
#include <sched.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <atomic>
#include <condition_variable>
#include <functional>
#include <mutex>
#include <stdexcept>
#include <thread>
#include <vector>

#if defined(__x86_64__)
#include <emmintrin.h>
#endif

#include "../../include/piplib_b200.h"
#include "pip_convert.h"
#include "pip_decode.h"
#include "pip_engine.h"
#include "pip_kernels.h"
#include "pip_segments.h"

typedef long long I;

static_assert(sizeof(PipProblemInfo_dp) == 32 && sizeof(PipInfo) == sizeof(PipProblemInfo_dp), "report layouts must agree");
static_assert(PIP_INFO_FLAG_WRAPPED == PIP_FLAG_WRAPPED, "report flags must agree");

namespace {

enum { S_SHIFT = 1, S_NEGATE = 2, S_REMOVE = 4, S_DUAL = 8 };   /* source/sol.h:35-48 */

I gcd_abs(I a, I b)
{
  unsigned long long x = a < 0 ? 0ull - (unsigned long long)a : (unsigned long long)a;
  unsigned long long y = b < 0 ? 0ull - (unsigned long long)b : (unsigned long long)b;
  while (y) { unsigned long long r = x % y; x = y; y = r; }
  return (I)x;
}

void *xmalloc(size_t n)
{
  void *p = malloc(n ? n : 1);
  if (!p) { fprintf(stderr, "Memory Overflow.\n"); exit(1); }
  return p;
}

/* what pip_solve derives from (domain, context, Bg, options) before any tableau exists,
 * source/piplib.c:758-797 */
struct Shape {
  int Np, Nn, Nl, Nm, Bg, Shift, Urs, sol_flags, nq, flags;
  bool has_ctx;
};

struct MatView { int rows, cols; const I *const *row; const I *dense; };
inline I MV(const MatView &m, int i, int j) { return m.row ? m.row[i][j] : m.dense[(size_t)i * m.cols + j]; }

/* the part that depends on the dimensions and the options only (Nl / Nm are left 0) */
Shape derive_shape_dims(int dom_cols, const MatView *ctx, int Bg, const PipOptions_dp &o)
{
  Shape s;
  memset(&s, 0, sizeof s);
  s.has_ctx = ctx != nullptr;
  s.Np = ctx ? ctx->cols - 2 : 0;
  s.Nn = dom_cols - s.Np - 2;
  if (o.Maximize) { s.sol_flags |= S_SHIFT | S_NEGATE; s.Shift = 1; }
  else if (o.Urs_unknowns) { s.sol_flags |= S_SHIFT; s.Shift = -1; }
  if (o.Urs_parms) { s.Urs = s.Np - (Bg >= 0); s.Np += s.Urs; }
  if (o.Maximize || o.Urs_unknowns)
    if (Bg < 0) { Bg = dom_cols - 1; s.Np++; s.sol_flags |= S_REMOVE; }
  s.Bg = Bg;
  s.nq = o.Nq;
  s.flags = 0;
  if (o.Nq) s.flags |= PIP_F_INT;
  else if (o.Compute_dual) { s.flags |= PIP_F_DUAL; s.sol_flags |= S_DUAL; }
  if (o.Deepest_cut) s.flags |= PIP_F_DEEPEST;
  return s;
}

Shape derive_shape(const MatView &dom, const MatView *ctx, int Bg, const PipOptions_dp &o)
{
  Shape s = derive_shape_dims(dom.cols, ctx, Bg, o);
  s.Nl = dom.rows;                      /* an equality becomes two tableau rows, source/tab.c:327-337 */
  for (int i = 0; i < dom.rows; i++) if (MV(dom, i, 0) == 0) s.Nl++;
  s.Nm = 0;
  if (ctx) { s.Nm = ctx->rows; for (int i = 0; i < ctx->rows; i++) if (MV(*ctx, i, 0) == 0) s.Nm++; }
  return s;
}

/* tab_Matrix2Tableau_xx (source/tab.c:292-393) writing `width`-wide rows to out: the per-row body is
 * pip_convert_row (pip_convert.h), shared with the device-side conversion kernel.
 * ctx_mode: the matrix is the context (n == -1 in the reference). */
/* returns false when some value does not fit the element type T */
template <class T>
bool matrix_to_rows(const MatView &mx, T *out, int width, int Nv, bool ctx_mode, int Shift, int Bg, int Urs)
{
  I lost = 0;
  int cur = 0;
  for (int i = 0; i < mx.rows; i++) {
    const I *in = mx.row ? mx.row[i] : mx.dense + (size_t)i * mx.cols;
    T *r = out + (size_t)cur * width;
    const bool ineq = pip_convert_row<T>(in, mx.cols, r, width, Nv, ctx_mode ? 1 : 0, Shift, Bg, Urs, lost);
    cur++;
    if (!ineq) { pip_convert_negate<T>(r, r + width, width, lost); cur++; }
  }
  return lost == 0;
}

/* words one problem contributes to the pool */
size_t problem_words(const Shape &s) { return (size_t)s.Nl * (s.Nn + s.Np + 1) + (size_t)s.Nm * (s.Np + 1); }

template <class T>
bool fill_problem(const MatView &dom, const MatView *ctx, const Shape &s, PipProblem &P, T *pool, size_t off)
{
  P.nvar = s.Nn; P.nparm = s.Np; P.ni = s.Nl; P.nc = s.Nm; P.bigparm = s.Bg; P.flags = s.flags; P.off = (I)off;
  if (s.sol_flags == 0 && s.Urs == 0) P.flags |= PIP_F_SIMPLE_SER;      /* decode without column surgery */
  T *tab = pool + off;
  bool ok = matrix_to_rows(dom, tab, s.Nn + s.Np + 1, s.Nn, false, s.Shift, s.Bg, s.Urs);
  if (ctx && s.Nm)
    ok = matrix_to_rows(*ctx, tab + (size_t)s.Nl * (s.Nn + s.Np + 1), s.Np + 1, s.Np - s.Urs, true, s.Shift, s.Bg - s.Nn - 1, s.Urs) && ok;
  return ok;
}

/* ---- cells -> tree: source/sol.c:435-734 ------------------------------------------------- */
/* cell accessors: the wire view (PipCellView) or a private unpacked copy (Simplify) */
struct ArrCells {
  const PipCell *c;
  int kind(int i) const { return c[i].kind; }
  I p1(int i) const { return c[i].p1; }
  I p2(int i) const { return c[i].p2; }
};

int skip_obj(const PipCell *c, int i);
int skip_new(const PipCell *c, int i) { return c[i].kind != PIP_C_NEW ? i : skip_obj(c, i + 1); }
int skip_obj(const PipCell *c, int i)
{
  while (c[i].kind == PIP_C_FREE || c[i].kind == PIP_C_ERROR) i++;
  switch (c[i].kind) {
  case PIP_C_NIL: case PIP_C_VAL: i++; break;
  case PIP_C_NEW: i = skip_new(c, i); break;
  case PIP_C_IF: i = skip_obj(c, i + 1); i = skip_obj(c, i); i = skip_obj(c, i); break;
  case PIP_C_LIST: case PIP_C_FORM: { int n = (int)c[i].p1; i++; while (n--) i = skip_obj(c, i); break; }
  case PIP_C_DIV: i = skip_obj(c, i + 1); i = skip_obj(c, i); break;
  }
  return skip_new(c, i);
}
/* sol_simplify_xx, source/sol.c:272-288 (works on a private copy of the cells) */
void simplify_cells(PipCell *c, int &ncell, int i)
{
  if (c[i].kind != PIP_C_IF) return;
  int j = skip_obj(c, i + 1), k = skip_obj(c, j);
  simplify_cells(c, ncell, k);
  simplify_cells(c, ncell, j);
  if (c[j].kind == PIP_C_NIL && c[k].kind == PIP_C_NIL) {
    c[i].kind = PIP_C_NIL;
    if (k >= ncell - 1) ncell = i + 1;
    else for (int l = i + 1; l <= k; l++) c[l].kind = PIP_C_FREE;
  }
}

template <class C>
PipVector_dp *decode_vector(const C &c, int *i, int Bg, int Urs_p, int flags)
{
  int n = (int)c.p1(*i), unbounded = 0;
  if (flags & S_REMOVE) --n;
  n -= Urs_p;
  const int first_urs = Urs_p + (Bg >= 0);
  PipVector_dp *v = (PipVector_dp *)xmalloc(sizeof *v);
  v->nb_elements = n;
  v->the_vector = (I *)xmalloc(sizeof(I) * (n > 0 ? n : 0));
  v->the_deno = (I *)xmalloc(sizeof(I) * (n > 0 ? n : 0));
  for (int j = 0, k = 0; k < n; j++) {
    (*i)++;
    I N = c.p1(*i), D = c.p2(*i), d = gcd_abs(N, D);
    if ((flags & S_SHIFT) && j == Bg) { N -= D; if (N != 0) unbounded = 1; }
    if ((flags & S_REMOVE) && j == Bg) continue;
    if (first_urs <= j && j < first_urs + Urs_p) continue;
    v->the_vector[k] = d ? N / d : 0;
    if (flags & S_NEGATE) v->the_vector[k] = -v->the_vector[k];
    v->the_deno[k] = (d == D) ? 1 : (d ? D / d : 0);
    k++;
  }
  if (unbounded) for (int k = 0; k < n; k++) v->the_deno[k] = 0;
  (*i)++;
  return v;
}

template <class C>
PipQuast_dp *decode_quast(const C &c, int *i, PipQuast_dp *father, int Bg, int Urs_p, int flags)
{
  while (c.kind(*i) == PIP_C_FREE) (*i)++;
  PipQuast_dp *q = (PipQuast_dp *)xmalloc(sizeof *q);
  q->newparm = nullptr; q->list = nullptr; q->condition = nullptr;
  q->next_then = q->next_else = nullptr; q->father = father;
  PipNewparm_dp *last = nullptr;
  while (c.kind(*i) == PIP_C_NEW) {                  /* sol_newparm_edit_xx, source/sol.c:525-577 */
    const int newcell = *i;
    (*i) += 2;
    PipNewparm_dp *np = (PipNewparm_dp *)xmalloc(sizeof *np);
    np->vector = decode_vector(c, i, Bg, Urs_p, flags & S_REMOVE);
    np->rank = (int)c.p1(newcell);
    np->deno = c.p1(*i);
    if (flags & S_REMOVE) np->rank--;
    np->rank -= Urs_p;
    np->next = nullptr;
    if (last) last->next = np; else q->newparm = np;
    last = np;
    (*i)++;
  }
  const int kind = c.kind(*i);
  const int nb = (int)c.p1(*i);
  (*i)++;
  if (kind == PIP_C_LIST) {                           /* sol_list_edit_xx, source/sol.c:591-638 */
    PipList_dp *head = (PipList_dp *)xmalloc(sizeof *head), *cur = head;
    head->next = nullptr; head->vector = nullptr;
    if (nb > 0) {
      head->vector = decode_vector(c, i, Bg, Urs_p, flags);
      for (int e = 1; e < nb; e++) {
        PipList_dp *l = (PipList_dp *)xmalloc(sizeof *l);
        l->vector = decode_vector(c, i, Bg, Urs_p, flags);
        l->next = nullptr;
        cur->next = l; cur = l;
      }
    }
    q->list = head;
    if (flags & S_DUAL) q->next_then = decode_quast(c, i, q, Bg, Urs_p, 0);
  } else if (kind == PIP_C_NIL) {
  } else if (kind == PIP_C_IF) {
    q->condition = decode_vector(c, i, Bg, Urs_p, flags & S_REMOVE);
    q->next_then = decode_quast(c, i, q, Bg, Urs_p, flags);
    q->next_else = decode_quast(c, i, q, Bg, Urs_p, flags);
  } else {
    fprintf(stderr, "\nAie !!! Flag %d inattendu.\n", kind);
    exit(1);
  }
  return q;
}

/* serialisation (the word format of oracle/ref_harness.c) */
struct Ser { I *out; long cap, len; unsigned long long h; bool hashing; };
inline void sput(Ser &s, I v)
{
  if (s.hashing) s.h += pip_hash_word((unsigned long long)v, (unsigned long long)s.len);
  if (s.out && s.len < s.cap) s.out[s.len] = v;
  s.len++;
}
void ser_vec(Ser &s, const PipVector_dp *v)
{
  sput(s, v->nb_elements);
  for (int i = 0; i < v->nb_elements; i++) { sput(s, v->the_vector[i]); sput(s, v->the_deno[i]); }
}
void ser_quast(Ser &s, const PipQuast_dp *q)
{
  if (!q) { sput(s, -1); return; }
  long n = 0;
  for (const PipNewparm_dp *np = q->newparm; np; np = np->next) n++;
  sput(s, n);
  for (const PipNewparm_dp *np = q->newparm; np; np = np->next) { sput(s, np->rank); sput(s, np->deno); ser_vec(s, np->vector); }
  if (q->condition) { sput(s, 2); ser_vec(s, q->condition); ser_quast(s, q->next_then); ser_quast(s, q->next_else); }
  else if (q->list) {
    sput(s, 1);
    n = 0; for (const PipList_dp *l = q->list; l; l = l->next) n++;
    sput(s, n);
    for (const PipList_dp *l = q->list; l; l = l->next) { sput(s, l->vector != nullptr); if (l->vector) ser_vec(s, l->vector); }
    sput(s, q->next_then != nullptr);
    if (q->next_then) ser_quast(s, q->next_then);
  } else sput(s, 0);
}

const char *fatal_message(int status)
{
  switch (status) {
  case PIP_ST_FATAL + 1: return "Integer overflow\n";
  case PIP_ST_FATAL + 2: return "Too much parameters\n";
  case PIP_ST_FATAL + 3: return "Too many variables\n";
  case PIP_ST_FATAL + 26: return "The solution is too complex! : sol\n";
  case PIP_ST_FAULT: return "Floating point exception\n";
  case PIP_ST_CAPACITY: return "piplib-b200: problem exceeds the largest device size class\n";
  case PIP_ST_UNSUPPORTED: return "piplib-b200: option not implemented on the device (Compute_dual / Deepest_cut)\n";
  }
  return "piplib-b200: solver error\n";
}

/* statistics of the last batch call: written and read under g_stats_mu (callers may solve from
 * several threads) */
PipBatchStats_dp g_stats;
std::mutex g_stats_mu;
void publish_stats(const PipBatchStats_dp &s) { std::lock_guard<std::mutex> g(g_stats_mu); g_stats = s; }

/* add one engine run to a statistics record (the per-problem counters are summed, not kept) */
void accumulate(PipBatchStats_dp &s, const PipBatchOut &out)
{
  for (const PipResult &r : out.res) {
    s.cells += (unsigned long long)r.ncells;
    s.pivots += r.pivots; s.cuts += r.cuts; s.subsolves += r.subsolves; s.splits += r.splits;
    s.elem_updates += ((unsigned long long)r.elem_updates_hi << 32) | r.elem_updates_lo;
    s.max_rows = std::max(s.max_rows, r.max_rows);
    s.max_cols = std::max(s.max_cols, r.max_cols);
    if (r.rflags & PIP_RES_WRAPPED) s.wrapped++;
  }
  s.seconds_h2d += out.times.h2d; s.seconds_kernel += out.times.kernel; s.seconds_d2h += out.times.d2h;
  s.launches += out.times.launches; s.rounds += out.times.rounds;
  s.device_ms += out.times.device_ms;
  s.h2d_bytes += out.times.h2d_bytes; s.d2h_bytes += out.times.d2h_bytes;
  for (int k = 0; k < PIP_NPHASE && k < 16; k++) s.phase_cycles[k] += out.times.phase_cycles[k];
}
void merge_stats(PipBatchStats_dp &s, const PipBatchStats_dp &o)
{
  s.cells += o.cells; s.pivots += o.pivots; s.cuts += o.cuts; s.subsolves += o.subsolves; s.splits += o.splits;
  s.elem_updates += o.elem_updates;
  s.wrapped += o.wrapped;
  s.max_rows = std::max(s.max_rows, o.max_rows); s.max_cols = std::max(s.max_cols, o.max_cols);
  s.seconds_h2d += o.seconds_h2d; s.seconds_kernel += o.seconds_kernel; s.seconds_d2h += o.seconds_d2h;
  s.launches += o.launches; s.rounds += o.rounds; s.device_ms += o.device_ms;
  s.h2d_bytes += o.h2d_bytes; s.d2h_bytes += o.d2h_bytes;
  for (int k = 0; k < 16; k++) s.phase_cycles[k] += o.phase_cycles[k];
}

thread_local std::vector<unsigned> t_last_flags;     /* pip_last_batch_flags_dp */

void account(const PipBatchOut &out, double host_seconds)
{
  t_last_flags.resize(out.res.size());
  for (size_t i = 0; i < out.res.size(); i++) t_last_flags[i] = (out.res[i].rflags & PIP_RES_WRAPPED) ? PIP_FLAG_WRAPPED : 0u;
  PipBatchStats_dp s;
  memset(&s, 0, sizeof s);
  accumulate(s, out);
  s.seconds_host = host_seconds;
  publish_stats(s);
}

/* ---- host threads: one persistent pool per process -----------------------------------------------
 * Size = the cores this process may use (sched_getaffinity) divided by the ranks that share the node
 * (LOCAL_WORLD_SIZE, set by torchrun / mpirun wrappers; PIPLIB_B200_THREADS overrides): 8 ranks on a
 * 32-core box get 4 workers each instead of 8 x 64 threads fighting for 32 cores.  Workers are created
 * once and parked on a condition variable; a parallel region hands out index ranges through an atomic
 * counter and the caller works too. */
class HostPool {
 public:
  /* never destroyed: the workers are detached and parked on the condition variable for the life of the
   * process (destroying a condition variable with waiters blocks in glibc -- the process would hang at exit) */
  static HostPool &get() { static HostPool *p = new HostPool; return *p; }
  size_t size() const { return nworkers_ + 1; }
  /* f(range index, begin, end) over `parts` nearly equal ranges of [0, n) */
  template <class F>
  void ranges(size_t n, size_t parts, F f)
  {
    parts = std::max<size_t>(1, std::min(parts, (n + 63) / 64));
    const size_t per = (n + parts - 1) / parts;
    if (parts == 1 || nworkers_ == 0) {
      for (size_t t = 0; t < parts; t++) { const size_t a = t * per, b = std::min(n, a + per); if (a < b) f(t, a, b); }
      return;
    }
    Job job;
    job.parts = parts;
    job.run = [&](size_t t) { const size_t a = t * per, b = std::min(n, a + per); if (a < b) f(t, a, b); };
    {
      std::lock_guard<std::mutex> g(mu_);
      jobs_.push_back(&job);
      job.active = 1;                   /* the caller takes ranges too */
    }
    cv_.notify_all();
    work_on(job);
    std::unique_lock<std::mutex> lk(mu_);
    /* the job lives on this stack: wait until every range is done AND no worker still holds the pointer */
    job.done_cv.wait(lk, [&] { return job.finished == job.parts && job.active == 0; });
    jobs_.erase(std::find(jobs_.begin(), jobs_.end(), &job));
  }

 private:
  struct Job {
    size_t parts = 0;
    std::atomic<size_t> next{0};
    size_t finished = 0;                /* under mu_ */
    int active = 0;                     /* threads inside work_on for this job, under mu_ */
    std::function<void(size_t)> run;
    std::condition_variable done_cv;
  };
  HostPool()
  {
    size_t cores = 1;
    cpu_set_t set;
    CPU_ZERO(&set);
    if (sched_getaffinity(0, sizeof set, &set) == 0) cores = std::max(1, CPU_COUNT(&set));
    else cores = std::max(1u, std::thread::hardware_concurrency());
    size_t share = 1;
    if (const char *lw = getenv("LOCAL_WORLD_SIZE")) share = std::max(1, atoi(lw));
    size_t want = std::max<size_t>(1, cores / share);
    if (const char *t = getenv("PIPLIB_B200_THREADS")) if (atoi(t) > 0) want = (size_t)atoi(t);
    nworkers_ = want > 1 ? want - 1 : 0;
    for (size_t i = 0; i < nworkers_; i++) std::thread([this] { worker(); }).detach();
  }
  void work_on(Job &job)
  {
    size_t mine = 0;
    for (;;) {
      const size_t t = job.next.fetch_add(1);
      if (t >= job.parts) break;
      job.run(t);
      mine++;
    }
    std::lock_guard<std::mutex> g(mu_);
    job.finished += mine;
    job.active--;
    if (job.finished == job.parts && job.active == 0) job.done_cv.notify_all();
  }
  void worker()
  {
    for (;;) {
      Job *job = nullptr;
      {
        std::unique_lock<std::mutex> lk(mu_);
        cv_.wait(lk, [&] {
          for (Job *j : jobs_) if (j->next.load() < j->parts) { job = j; return true; }
          return false;
        });
        job->active++;
      }
      work_on(*job);
    }
  }
  std::mutex mu_;
  std::condition_variable cv_;
  std::vector<Job *> jobs_;
  size_t nworkers_ = 0;
};

template <class F>
void parallel_for(size_t n, F f)
{
  HostPool::get().ranges(n, HostPool::get().size(), [&](size_t, size_t a, size_t b) { f(a, b); });
}

const PipOptions_dp DEFAULT_OPTIONS = {1, 0, 0, 0, 0, 0, 0, 0};

}  // namespace

extern "C" {

/* ---- reference API ------------------------------------------------------------------------ */
void pip_init_dp(void) {}
void pip_close_dp(void) {}

PipOptions_dp *pip_options_init_dp(void)
{
  PipOptions_dp *o = (PipOptions_dp *)xmalloc(sizeof *o);
  *o = DEFAULT_OPTIONS;
  return o;
}
void pip_options_free_dp(PipOptions_dp *o) { free(o); }
void pip_options_print_dp(FILE *f, PipOptions_dp *o)
{
  fprintf(f, "Option setting is:\n");
  fprintf(f, "Nq          =%d\n", o->Nq);
  fprintf(f, "Verbose     =%d\n", o->Verbose);
  fprintf(f, "Simplify    =%d\n", o->Simplify);
  fprintf(f, "Deepest_cut =%d\n", o->Deepest_cut);
  fprintf(f, "Maximize    =%d\n", o->Maximize);
  fprintf(f, "Urs_parms   =%d\n", o->Urs_parms);
  fprintf(f, "Urs_unknowns=%d\n", o->Urs_unknowns);
  fprintf(f, "\n");
}

PipMatrix_dp *pip_matrix_alloc_dp(unsigned rows, unsigned cols)
{
  PipMatrix_dp *m = (PipMatrix_dp *)xmalloc(sizeof *m);
  m->NbRows = rows; m->NbColumns = cols; m->p_Init_size = (int)(rows * cols);
  m->p = nullptr; m->p_Init = nullptr;
  if (rows && cols) {
    m->p = (I **)xmalloc(sizeof(I *) * rows);
    m->p_Init = (I *)xmalloc(sizeof(I) * (size_t)rows * cols);
    memset(m->p_Init, 0, sizeof(I) * (size_t)rows * cols);
    for (unsigned i = 0; i < rows; i++) m->p[i] = m->p_Init + (size_t)i * cols;
  }
  return m;
}
void pip_matrix_free_dp(PipMatrix_dp *m)
{
  if (!m) return;
  free(m->p_Init); free(m->p); free(m);
}
void pip_matrix_print_dp(FILE *f, PipMatrix_dp *m)
{
  fprintf(f, "%d %d\n", m->NbRows, m->NbColumns);
  for (unsigned i = 0; i < m->NbRows; i++) {
    for (unsigned j = 0; j < m->NbColumns; j++) fprintf(f, " %lld", m->p[i][j]);
    fprintf(f, "\n");
  }
}
/* pip_matrix_read_xx, source/piplib.c:576-619: '#' comment lines, "rows cols", then one row per line */
PipMatrix_dp *pip_matrix_read_dp(FILE *f)
{
  char s[1024];
  unsigned rows = 0, cols = 0;
  for (;;) {
    if (!fgets(s, sizeof s, f)) { fprintf(stderr, "Not enough rows.\n"); exit(1); }
    if (*s == '#' || *s == '\n') continue;
    if (sscanf(s, " %u %u", &rows, &cols) >= 2) break;
  }
  PipMatrix_dp *m = pip_matrix_alloc_dp(rows, cols);
  for (unsigned i = 0; i < rows; i++) {
    char *c;
    for (;;) {
      if (!fgets(s, sizeof s, f)) { fprintf(stderr, "Not enough rows.\n"); exit(1); }
      c = s;
      while (isspace((unsigned char)*c) && *c != '\n') c++;
      if (*c != '#' && *c != '\n' && *c != 0) break;
    }
    for (unsigned j = 0; j < cols; j++) {
      char tok[1024]; int used = 0;
      if (*c == 0 || *c == '#' || *c == '\n' || sscanf(c, "%1023s%n", tok, &used) < 1) {
        fprintf(stderr, "Not enough columns.\n"); exit(1);
      }
      long long v = 0; sscanf(tok, "%lld", &v);
      m->p[i][j] = v;
      c += used;
    }
  }
  return m;
}

void pip_vector_print_dp(FILE *f, PipVector_dp *v)
{
  if (!v) return;
  fprintf(f, "#[");
  for (int i = 0; i < v->nb_elements; i++) {
    fprintf(f, " %lld", v->the_vector[i]);
    if (v->the_deno[i] != 1) fprintf(f, "/%lld", v->the_deno[i]);
  }
  fprintf(f, "]");
}
void pip_newparm_print_dp(FILE *f, PipNewparm_dp *np, int indent)
{
  for (; np; np = np->next) {
    for (int i = 0; i < indent; i++) fprintf(f, " ");
    fprintf(f, "(newparm %d (div ", np->rank);
    pip_vector_print_dp(f, np->vector);
    fprintf(f, " %lld))\n", np->deno);
  }
}
void pip_list_print_dp(FILE *f, PipList_dp *l, int indent)
{
  for (int i = 0; i < indent; i++) fprintf(f, " ");
  if (!l) { fprintf(f, "()\n"); return; }
  fprintf(f, "(list\n");
  for (; l; l = l->next)
    if (l->vector) {
      for (int i = 0; i < indent + 1; i++) fprintf(f, " ");
      pip_vector_print_dp(f, l->vector);
      fprintf(f, "\n");
    }
  for (int i = 0; i < indent; i++) fprintf(f, " ");
  fprintf(f, ")\n");
}
void pip_quast_print_dp(FILE *f, PipQuast_dp *q, int indent)
{
  const int ni = indent >= 0 ? indent + 1 : indent;
  if (!q) { for (int i = 0; i < indent; i++) fprintf(f, " "); fprintf(f, "void\n"); return; }
  pip_newparm_print_dp(f, q->newparm, indent);
  if (!q->condition) {
    pip_list_print_dp(f, q->list, indent);
    if (q->next_then) pip_quast_print_dp(f, q->next_then, ni);
  } else {
    for (int i = 0; i < indent; i++) fprintf(f, " ");
    fprintf(f, "(if ");
    pip_vector_print_dp(f, q->condition);
    fprintf(f, "\n");
    pip_quast_print_dp(f, q->next_then, ni);
    pip_quast_print_dp(f, q->next_else, ni);
    for (int i = 0; i < indent; i++) fprintf(f, " ");
    fprintf(f, ")\n");
  }
}

void pip_vector_free_dp(PipVector_dp *v) { if (v) { free(v->the_vector); free(v->the_deno); free(v); } }
void pip_newparm_free_dp(PipNewparm_dp *np)
{
  while (np) { PipNewparm_dp *n = np->next; pip_vector_free_dp(np->vector); free(np); np = n; }
}
void pip_list_free_dp(PipList_dp *l)
{
  while (l) { PipList_dp *n = l->next; pip_vector_free_dp(l->vector); free(l); l = n; }
}
void pip_quast_free_dp(PipQuast_dp *q)
{
  if (!q) return;
  pip_newparm_free_dp(q->newparm);
  pip_list_free_dp(q->list);
  pip_vector_free_dp(q->condition);
  pip_quast_free_dp(q->next_then);
  pip_quast_free_dp(q->next_else);
  free(q);
}

long pip_quast_serialize_dp(const PipQuast_dp *q, long long *out, long cap)
{
  Ser s = {out, cap, 0, 0, false};
  ser_quast(s, q);
  return s.len;
}

int pip_set_device_dp(int device) { return PipEngine::get().set_device(device); }
void pip_set_donation_dp(int mode) { pip_engine_set_donation(mode < 0 ? -1 : mode > 0 ? 1 : 0); }
const char *pip_b200_version(void) { return "piplib-b200 0.1 (sm_100a)"; }
long long pip_last_batch_flags_dp(unsigned *flags, long long cap)
{
  const long long n = (long long)t_last_flags.size();
  for (long long i = 0; i < n && i < cap && flags; i++) flags[i] = t_last_flags[i];
  return n;
}
void pip_last_batch_stats_dp(PipBatchStats_dp *out)
{
  if (!out) return;
  std::lock_guard<std::mutex> g(g_stats_mu);
  *out = g_stats;
}

/* ---- batch entry points -------------------------------------------------------------------- */

static void unpack_cells(const PipCellView &v, std::vector<PipCell> &out)
{
  out.resize(v.n);
  for (int i = 0; i < v.n; i++) { out[i].kind = v.kind(i); out[i].pad = 0; out[i].p1 = v.p1(i); out[i].p2 = v.p2(i); }
}

/* pip_quast_equalities_dual_xx, source/piplib.c:651-690: an equality was solved as a pair of
 * inequalities; keep one dual value per equality (negated when it belongs to the negative half) */
static void equalities_dual(PipQuast_dp *sol, const MatView &dom)
{
  if (!sol) return;
  if (sol->condition) { equalities_dual(sol->next_then, dom); equalities_dual(sol->next_else, dom); }
  if (!sol->list || !sol->next_then || !sol->next_then->list) return;
  PipList_dp **lp = &sol->next_then->list;
  for (int i = 0; i < dom.rows; i++) {
    if (MV(dom, i, 0) != 0) { lp = &(*lp)->next; continue; }
    if ((*lp)->vector->the_vector[0] != 0) {
      lp = &(*lp)->next;
      PipList_dp *l = *lp;
      *lp = l->next; l->next = nullptr;
      pip_list_free_dp(l);
    } else {
      PipList_dp *l = *lp;
      *lp = l->next; l->next = nullptr;
      pip_list_free_dp(l);
      (*lp)->vector->the_vector[0] = -(*lp)->vector->the_vector[0];
      lp = &(*lp)->next;
    }
  }
}

/* the reference keeps the cells of the last solve in its global sol_space until the next solve
 * (source/sol.c:54-55), which is what the exported sol_quast_edit_xx reads; ours is per thread and
 * holds the cells of the last pip_solve_dp / batch-of-one on this thread (pip_cells_bind_dp binds
 * any other stream) */
static thread_local std::vector<PipCell> t_sol_space;

static PipQuast_dp *decode_one(const PipBatchOut &bo, size_t i, const Shape &s, int simplify)
{
  const PipCellView v = bo.cells_of(i);
  int at = 0;
  if (simplify) {
    std::vector<PipCell> copy;
    unpack_cells(v, copy);
    int n = v.n;
    simplify_cells(copy.data(), n, 0);
    ArrCells a = {copy.data()};
    return decode_quast(a, &at, nullptr, s.Bg - s.Nn - 1, s.Urs, s.sol_flags);
  }
  return decode_quast(v, &at, nullptr, s.Bg - s.Nn - 1, s.Urs, s.sol_flags);
}

/* serialise problem i straight from its cells (status OK or VOID) with the decoder the device
 * uses too (pip_decode.h) */
static void serialize_one(const PipBatchOut &bo, size_t i, const Shape &s, int simplify, Ser &out,
                          const MatView *dom = nullptr)
{
  if (dom && (s.sol_flags & S_DUAL) && s.Nl > dom->rows && bo.res[i].status == PIP_ST_OK) {
    /* Compute_dual with equalities: the post-pass works on the tree (source/piplib.c:867-868) */
    PipQuast_dp *q = decode_one(bo, i, s, simplify);
    equalities_dual(q, *dom);
    ser_quast(out, q);
    pip_quast_free_dp(q);
    return;
  }
  PipSer ps = {out.out, out.cap, out.len, out.h, out.hashing ? 1 : 0, 0, 0};
  if (bo.res[i].status == PIP_ST_VOID) pip_sput(ps, -1);
  else {
    const PipCellView v = bo.cells_of(i);
    if (simplify) {
      std::vector<PipCell> copy;
      unpack_cells(v, copy);
      int n = v.n;
      simplify_cells(copy.data(), n, 0);
      PipRawCells a = {copy.data()};
      pip_ser_cells(ps, a, n, s.Bg - s.Nn - 1, s.Urs, s.sol_flags);
    } else pip_ser_cells(ps, v, v.n, s.Bg - s.Nn - 1, s.Urs, s.sol_flags);
  }
  out.len = (long)ps.len; out.h = ps.h;
}

int pip_solve_batch_dp(int n, PipMatrix_dp *const *domains, PipMatrix_dp *const *contexts,
                       const int *bignums, const PipOptions_dp *options, PipQuast_dp **out, int *status)
{
  if (n <= 0) return 0;
  const PipOptions_dp &o = options ? *options : DEFAULT_OPTIONS;
  /* one batch call at a time: it stages in the engine's pinned buffers and decodes from them
   * (the reference is not re-entrant either: sol_space and the cross counters are globals) */
  static std::mutex batch_mu;
  std::lock_guard<std::mutex> batch_guard(batch_mu);
  try {
    std::vector<Shape> shapes(n);
    std::vector<PipProblem> prob(n);
    std::vector<size_t> off(n + 1, 0);
    std::vector<int> live;            /* problems that reach the device */
    for (int i = 0; i < n; i++) {
      out[i] = nullptr;
      if (!domains[i]) { status[i] = PIP_STATUS_VOID; off[i + 1] = off[i]; continue; }
      MatView d = {(int)domains[i]->NbRows, (int)domains[i]->NbColumns, domains[i]->p, nullptr};
      MatView c, *cp = nullptr;
      if (contexts && contexts[i]) { c = {(int)contexts[i]->NbRows, (int)contexts[i]->NbColumns, contexts[i]->p, nullptr}; cp = &c; }
      shapes[i] = derive_shape(d, cp, bignums ? bignums[i] : -1, o);
      off[i + 1] = off[i] + problem_words(shapes[i]);
      live.push_back(i);
    }
    /* the tableaux go straight into the engine's pinned staging area, as int32 when every value fits (the
     * shared-memory int32 class is the fast one), else as int64 */
    PipEngine &E = PipEngine::get();
    void *pool = E.pinned_input((off[n] + 8) << 3);
    std::vector<PipProblem> lp(live.size());
    auto fill_all = [&](auto *typed) -> bool {
      std::atomic<int> lost(0);
      parallel_for(live.size(), [&](size_t a, size_t b) {
        bool good = true;
        for (size_t q = a; q < b; q++) {
          int i = live[q];
          MatView d = {(int)domains[i]->NbRows, (int)domains[i]->NbColumns, domains[i]->p, nullptr};
          MatView c, *cp = nullptr;
          if (contexts && contexts[i]) { c = {(int)contexts[i]->NbRows, (int)contexts[i]->NbColumns, contexts[i]->p, nullptr}; cp = &c; }
          good = fill_problem(d, cp, shapes[i], lp[q], typed, off[i]) && good;
        }
        if (!good) lost.store(1);
      });
      return lost.load() == 0;
    };
    int elem_log2 = 2;
    if (getenv("PIPLIB_B200_NO_INT32") || !fill_all((int *)pool)) { elem_log2 = 3; fill_all((I *)pool); }
    /* same shape everywhere (the usual batch: one loop nest, many parameter samples): planned once */
    bool same = !live.empty();
    for (size_t q = 1; q < live.size() && same; q++) {
      const PipProblem &A = lp[0], &B = lp[q];
      same = A.nvar == B.nvar && A.nparm == B.nparm && A.ni == B.ni && A.nc == B.nc && A.bigparm == B.bigparm && A.flags == B.flags;
    }
    PipProblem shape0;
    PipBatchIn in;
    in.n = live.size(); in.h_prob = lp.data(); in.h_pool = pool; in.pool_words = off[n]; in.elem_log2 = elem_log2;
    if (same) { shape0 = lp[0]; shape0.off = 0; in.uniform = &shape0; }
    PipBatchOut bo;
    PipEngine::get().run(in, bo);
    double t0 = 0;
    {
      struct timespec ts; clock_gettime(CLOCK_MONOTONIC, &ts); t0 = ts.tv_sec + 1e-9 * ts.tv_nsec;
    }
    parallel_for(live.size(), [&](size_t a, size_t b) {
      for (size_t q = a; q < b; q++) {
        int i = live[q];
        status[i] = bo.res[q].status;
        if (status[i] == PIP_ST_OK) {
          if (n == 1) {
            unpack_cells(bo.cells_of(q), t_sol_space);
            int nc1 = (int)t_sol_space.size();
            if (o.Simplify && nc1) { simplify_cells(t_sol_space.data(), nc1, 0); t_sol_space.resize(nc1); }
          }
          out[i] = decode_one(bo, q, shapes[i], o.Simplify);
          if ((shapes[i].sol_flags & S_DUAL) && shapes[i].Nl > (int)domains[i]->NbRows) {
            MatView d = {(int)domains[i]->NbRows, (int)domains[i]->NbColumns, domains[i]->p, nullptr};
            equalities_dual(out[i], d);
          }
        }
      }
    });
    {
      struct timespec ts; clock_gettime(CLOCK_MONOTONIC, &ts);
      account(bo, ts.tv_sec + 1e-9 * ts.tv_nsec - t0);
    }
  } catch (const std::exception &e) {
    fprintf(stderr, "%s\n", e.what());
    return -1;
  }
  return 0;
}

PipQuast_dp *pip_solve_dp(PipMatrix_dp *domain, PipMatrix_dp *context, int Bg, PipOptions_dp *options)
{
  if (!domain) return nullptr;
  PipQuast_dp *q = nullptr;
  int status = 0;
  PipMatrix_dp *doms[1] = {domain}, *ctxs[1] = {context};
  int bgs[1] = {Bg};
  if (pip_solve_batch_dp(1, doms, ctxs, bgs, options, &q, &status) != 0) exit(1);
  if (status == PIP_ST_OK || status == PIP_ST_VOID) return q;
  /* the reference reports every error with a message and exit(code) (SURVEY.md section 5) */
  fputs(fatal_message(status), stderr);
  exit(status >= PIP_ST_FATAL && status < PIP_ST_FAULT ? status - PIP_ST_FATAL : 1);
}

int pip_traiter_batch_dp(int n, const PipTableauHeader_dp *hdr, const long long *const *tab,
                         const long long *const *ctx, int *status, PipCell_dp *cells_out,
                         long long cell_cap, long long *cell_off, int *ncells, long long *cells_needed)
{
  if (n <= 0) return 0;
  try {
    std::vector<PipProblem> prob(n);
    std::vector<size_t> off(n + 1, 0);
    for (int i = 0; i < n; i++) {
      const PipTableauHeader_dp &h = hdr[i];
      off[i + 1] = off[i] + (size_t)h.ni * (h.nvar + h.nparm + 1) + (size_t)h.nc * (h.nparm + 1);
    }
    std::vector<I> pool(off[n] + 1);
    for (int i = 0; i < n; i++) {
      const PipTableauHeader_dp &h = hdr[i];
      size_t tw = (size_t)h.ni * (h.nvar + h.nparm + 1), cw = (size_t)h.nc * (h.nparm + 1);
      if (tw) memcpy(pool.data() + off[i], tab[i], tw * sizeof(I));
      if (cw) memcpy(pool.data() + off[i] + tw, ctx[i], cw * sizeof(I));
      PipProblem &P = prob[i];
      P.nvar = h.nvar; P.nparm = h.nparm; P.ni = h.ni; P.nc = h.nc; P.bigparm = h.bigparm;
      P.flags = ((h.nq & 1) ? PIP_F_INT : (h.nq & 2) ? PIP_F_DUAL : 0) | ((h.nq & 4) ? PIP_F_DEEPEST : 0);
      P.off = (I)off[i];
    }
    PipBatchIn in;
    in.n = n; in.h_prob = prob.data(); in.h_pool = pool.data(); in.pool_words = off[n];
    PipBatchOut bo;
    PipEngine::get().run(in, bo);
    long long total = 0;
    for (int i = 0; i < n; i++) total += bo.res[i].ncells;
    if (cells_needed) *cells_needed = total;
    long long at = 0;
    for (int i = 0; i < n; i++) {
      status[i] = bo.res[i].status;
      ncells[i] = bo.res[i].ncells;
      cell_off[i] = at;
      if (at + bo.res[i].ncells <= cell_cap && bo.res[i].ncells) {
        const PipCellView v = bo.cells_of(i);
        for (int k = 0; k < v.n; k++) {
          PipCell_dp &o = cells_out[at + k];
          o.kind = v.kind(k); o.pad = 0; o.p1 = v.p1(k); o.p2 = v.p2(k);
        }
      }
      at += bo.res[i].ncells;
    }
    account(bo, 0);
    if (total > cell_cap) return -2;
  } catch (const std::exception &e) {
    fprintf(stderr, "%s\n", e.what());
    return -1;
  }
  return 0;
}

/* sol_quast_edit_xx, include/piplib/piplib.h:398-402 / source/sol.c:664-734: decode the quast that
 * starts at cell *i of the current solution space (the cells of the last pip_solve_dp on this thread,
 * or the stream bound with pip_cells_bind_dp); *i is left behind the decoded object */
PipQuast_dp *sol_quast_edit_dp(int *i, PipQuast_dp *father, int Bg, int Urs_p, int flags)
{
  if (!i || *i < 0 || (size_t)*i >= t_sol_space.size()) return nullptr;
  ArrCells a = {t_sol_space.data()};
  return decode_quast(a, i, father, Bg, Urs_p, flags);
}
void pip_cells_bind_dp(const PipCell_dp *cells, int ncells)
{
  static_assert(sizeof(PipCell_dp) == sizeof(PipCell), "cell layouts must agree");
  t_sol_space.assign((const PipCell *)cells, (const PipCell *)cells + (ncells > 0 ? ncells : 0));
}

/* sol_simplify_xx (source/sol.c:272-288) on a problem's cells as returned by pip_traiter_batch_dp:
 * the `-z` option of the CLI.  Cells may become Free (kind 0); *ncells may shrink. */
void pip_cells_simplify_dp(PipCell_dp *cells, int *ncells)
{
  if (!cells || !ncells || *ncells <= 0) return;
  static_assert(sizeof(PipCell_dp) == sizeof(PipCell), "cell layouts must agree");
  simplify_cells((PipCell *)cells, *ncells, 0);
}

}  // extern "C"

/* ---- dense batches -------------------------------------------------------------------------- */
namespace {

double wall()
{
  struct timespec ts; clock_gettime(CLOCK_MONOTONIC, &ts);
  return ts.tv_sec + 1e-9 * ts.tv_nsec;
}

struct DenseArgs {
  long long n; int dr, dc; const I *dom; int has_ctx, cr, cc; const I *ctx; int bignum; PipOptions_dp opt;
};

/* one pipeline unit: problems [first, first + n) of a dense batch */
struct DenseChunk {
  size_t first = 0, n = 0;
  std::vector<Shape> shapes;
  std::vector<PipProblem> prob;
  std::vector<size_t> off;
  size_t pool_elems = 0;
  int elem_log2 = 3;
  PipBatchOut out;
  std::vector<std::vector<I>> bufs;     /* serialised words, one buffer per worker range */
  std::vector<long long> words;         /* per problem */
  size_t per = 0;                       /* problems per worker range */
};

unsigned host_threads() { return (unsigned)HostPool::get().size(); }

template <class F>
void parallel_ranges(size_t n, size_t nt, F f)
{
  HostPool::get().ranges(n, nt, f);
}

/* shapes + offsets of a chunk */
void plan_chunk(const DenseArgs &A, DenseChunk &C, size_t nthreads)
{
  const size_t n = C.n;
  C.shapes.resize(n);
  C.prob.resize(n);
  C.off.assign(n + 1, 0);
  parallel_ranges(n, nthreads, [&](size_t, size_t a, size_t b) {
    for (size_t i = a; i < b; i++) {
      const size_t g = C.first + i;
      MatView d = {A.dr, A.dc, nullptr, A.dom + g * A.dr * A.dc};
      MatView c = {A.cr, A.cc, nullptr, A.has_ctx ? A.ctx + g * A.cr * A.cc : nullptr};
      C.shapes[i] = derive_shape(d, A.has_ctx ? &c : nullptr, A.bignum, A.opt);
    }
  });
  for (size_t i = 0; i < n; i++) C.off[i + 1] = C.off[i] + problem_words(C.shapes[i]);
  C.pool_elems = C.off[n];
  C.elem_log2 = 3;
}

/* Optimistic plan without a pass over the inputs: every problem of a dense batch has the same
 * dimensions and options, so unless the number of equality rows varies (each becomes two tableau
 * rows, source/tab.c:327-337) every problem has the shape of the first one and offsets are
 * arithmetic.  convert_chunk_t checks the assumption problem by problem while the rows are in the
 * cache anyway and reports a mismatch; the caller then falls back to plan_chunk. */
void plan_chunk_uniform(const DenseArgs &A, DenseChunk &C)
{
  const size_t n = C.n, g = C.first;
  MatView d = {A.dr, A.dc, nullptr, A.dom + g * A.dr * A.dc};
  MatView c = {A.cr, A.cc, nullptr, A.has_ctx ? A.ctx + g * A.cr * A.cc : nullptr};
  const Shape s0 = derive_shape(d, A.has_ctx ? &c : nullptr, A.bignum, A.opt);
  const size_t w0 = problem_words(s0);
  C.shapes.assign(n, s0);
  C.prob.resize(n);
  C.off.resize(n + 1);
  for (size_t i = 0; i <= n; i++) C.off[i] = i * w0;
  C.pool_elems = C.off[n];
  C.elem_log2 = 3;
}

template <class T>
bool convert_chunk_t(const DenseArgs &A, DenseChunk &C, T *pool, size_t nthreads, std::atomic<int> *mismatch)
{
  std::vector<char> ok(nthreads + 1, 1);
  parallel_ranges(C.n, nthreads, [&](size_t t, size_t a, size_t b) {
    bool good = true;
    for (size_t i = a; i < b; i++) {
      const size_t g = C.first + i;
      MatView d = {A.dr, A.dc, nullptr, A.dom + g * A.dr * A.dc};
      MatView c = {A.cr, A.cc, nullptr, A.has_ctx ? A.ctx + g * A.cr * A.cc : nullptr};
      if (mismatch) {
        const Shape si = derive_shape(d, A.has_ctx ? &c : nullptr, A.bignum, A.opt);
        if (si.Nl != C.shapes[i].Nl || si.Nm != C.shapes[i].Nm) { mismatch->store(1); break; }
      }
      good = fill_problem(d, A.has_ctx ? &c : nullptr, C.shapes[i], C.prob[i], pool, C.off[i]) && good;
    }
    ok[t] = good;
  });
  for (char k : ok) if (!k) return false;
  return true;
}
/* Convert a chunk into the pinned staging area of `E`, trying the narrowest element first
 * (int8, then int32, then int64); `hint` remembers the width that worked for earlier chunks. */
void *convert_chunk(const DenseArgs &A, DenseChunk &C, PipEngine &E, size_t nthreads, std::atomic<int> *hint,
                    std::atomic<int> *mismatch = nullptr)
{
  int start = hint ? hint->load() : 0;
  void *pool = E.pinned_input((C.pool_elems + 8) << 3);
  for (int w = start;; w = (w == 0 ? 2 : 3)) {
    bool ok;
    if (w == 0) ok = convert_chunk_t(A, C, (signed char *)pool, nthreads, mismatch);
    else if (w == 2) ok = convert_chunk_t(A, C, (int *)pool, nthreads, mismatch);
    else ok = convert_chunk_t(A, C, (I *)pool, nthreads, mismatch);
    if (mismatch && mismatch->load()) return pool;
    if (ok || w == 3) {
      C.elem_log2 = w;
      if (hint && w > hint->load()) hint->store(w);
      return pool;
    }
  }
}

/* words ser_quast_direct would emit, without touching the values (structure only) */
template <class C>
long long len_vector(const C &c, int *i, int Bg, int Urs_p, int flags)
{
  int n = (int)c.p1(*i);
  if (flags & S_REMOVE) --n;
  n -= Urs_p;
  const int first_urs = Urs_p + (Bg >= 0);
  for (int j = 0, k = 0; k < n; j++) {
    (*i)++;
    if ((flags & S_REMOVE) && j == Bg) continue;
    if (first_urs <= j && j < first_urs + Urs_p) continue;
    k++;
  }
  (*i)++;
  return 1 + 2ll * (n > 0 ? n : 0);
}
template <class C>
long long len_quast(const C &c, int *i, int Bg, int Urs_p, int flags)
{
  while (c.kind(*i) == PIP_C_FREE) (*i)++;
  long long w = 1;
  while (c.kind(*i) == PIP_C_NEW) {
    (*i) += 2;
    w += 2 + len_vector(c, i, Bg, Urs_p, flags & S_REMOVE);
    (*i)++;
  }
  const int kind = c.kind(*i);
  const int nb = (int)c.p1(*i);
  (*i)++;
  w += 1;
  if (kind == PIP_C_LIST) {
    if (nb == 0) w += 2;
    else { w += 1; for (int e = 0; e < nb; e++) w += 1 + len_vector(c, i, Bg, Urs_p, flags); }
    w += 1;
    if (flags & S_DUAL) w += len_quast(c, i, Bg, Urs_p, 0);
  } else if (kind == PIP_C_IF) {
    w += len_vector(c, i, Bg, Urs_p, flags & S_REMOVE);
    w += len_quast(c, i, Bg, Urs_p, flags);
    w += len_quast(c, i, Bg, Urs_p, flags);
  }
  return w;
}

/* Serialise every solved problem of the chunk straight from its cells into the caller's stream.
 * Pass 1 sizes each problem (structure walk, no arithmetic); the chunk then reserves its span of
 * `ser` with one atomic add (chunks finish in any order, so spans are not in problem order);
 * pass 2 decodes in place, hashing on the fly. */
void emit_chunk(const DenseArgs &A, DenseChunk &C, int *status, unsigned long long *hashes,
                long long *ser, long long ser_cap, long long *ser_off, long long *ser_len,
                std::atomic<long long> *cursor, size_t nthreads, PipInfo *info = nullptr)
{
  const size_t n = C.n;
  const bool keep = ser != nullptr && ser_off != nullptr;
  const int simplify = A.opt.Simplify;
  for (size_t i = 0; i < n; i++) status[C.first + i] = C.out.res[i].status;
  if (info) for (size_t i = 0; i < n; i++) info[C.first + i] = pip_info_of(C.out.res[i]);
  if (!keep && !hashes) return;
  C.words.assign(n, 0);
  nthreads = std::max<size_t>(1, std::min(nthreads, (n + 63) / 64));
  const size_t per = (n + nthreads - 1) / nthreads;
  std::vector<long long> range_words(nthreads + 1, 0);
  if (keep) {
    parallel_ranges(n, nthreads, [&](size_t t, size_t a, size_t b) {
      long long sum = 0;
      for (size_t i = a; i < b; i++) {
        const int st = C.out.res[i].status;
        long long w = 0;
        if (st == PIP_ST_VOID) w = 1;
        else if (st == PIP_ST_OK) {
          const bool dualeq = (C.shapes[i].sol_flags & S_DUAL) && C.shapes[i].Nl > A.dr;
          if (simplify || dualeq) {
            MatView d = {A.dr, A.dc, nullptr, A.dom ? A.dom + (C.first + i) * A.dr * A.dc : nullptr};
            Ser s = {nullptr, 0, 0, 0, false};
            serialize_one(C.out, i, C.shapes[i], simplify, s, A.dom ? &d : nullptr);
            w = s.len;
          }
          else {
            const PipCellView v = C.out.cells_of(i);
            int at = 0;
            w = len_quast(v, &at, C.shapes[i].Bg - C.shapes[i].Nn - 1, C.shapes[i].Urs, C.shapes[i].sol_flags);
          }
        }
        C.words[i] = w;
        sum += w;
      }
      range_words[t] = sum;
    });
  }
  long long total = 0;
  std::vector<long long> range_base(nthreads + 1, 0);
  for (size_t t = 0; t < nthreads; t++) { range_base[t] = total; total += range_words[t]; }
  const long long base = keep ? cursor->fetch_add(total) : 0;
  const bool fits = keep && base + total <= ser_cap;
  parallel_ranges(n, nthreads, [&](size_t t, size_t a, size_t b) {
    long long at = base + range_base[t];
    for (size_t i = a; i < b; i++) {
      const int st = C.out.res[i].status;
      unsigned long long h = 0;
      if (st == PIP_ST_OK || st == PIP_ST_VOID) {
        Ser s = {fits ? ser + at : nullptr, fits ? (long)C.words[i] : 0, 0, 0xcbf29ce484222325ULL, hashes != nullptr};
        MatView d = {A.dr, A.dc, nullptr, A.dom ? A.dom + (C.first + i) * A.dr * A.dc : nullptr};
        if (fits || hashes) serialize_one(C.out, i, C.shapes[i], simplify, s, A.dom ? &d : nullptr);
        h = s.h;
      }
      if (hashes) hashes[C.first + i] = h;
      if (keep) { ser_off[C.first + i] = at; if (ser_len) ser_len[C.first + i] = C.words[i]; at += C.words[i]; }
    }
  });
  (void)per;
}

/* device-decode mode, results staged through pinned scratch (the caller's stream is pageable memory):
 * `words` = the chunk's compact buffer (int32 words where they fit), per-problem arrays in SoA form.
 * Reserve the chunk's span of the caller's stream and widen every problem's words into it. */
void emit_chunk_staged(size_t first, size_t n, const pip_i64 *words, const int *st, const pip_u64 *hs,
                       const long long *off, const long long *len, int *status, unsigned long long *hashes,
                       long long *ser, long long ser_cap, long long *ser_off, long long *ser_len,
                       std::atomic<long long> *cursor, size_t nthreads, std::vector<long long> &at)
{
  const bool keep = ser != nullptr && ser_off != nullptr;
  long long total = 0;
  at.resize(n);
  for (size_t i = 0; i < n; i++) { at[i] = total; total += len[i] & ~PIP_LEN_NARROW; }
  const long long base = keep ? cursor->fetch_add(total) : 0;
  const bool fits = keep && base + total <= ser_cap;
  parallel_ranges(n, nthreads, [&](size_t, size_t a, size_t b) {
    for (size_t i = a; i < b; i++) {
      const int s0 = st[i];
      status[first + i] = PIP_STATUS_IS_FINAL(s0) ? s0 : PIP_ST_CAPACITY;
      if (hashes) hashes[first + i] = hs[i];
      if (!keep) continue;
      const long long w = len[i] & ~PIP_LEN_NARROW;
      ser_off[first + i] = base + at[i];
      if (ser_len) ser_len[first + i] = w;
      if (!fits || !w) continue;
      I *dst = ser + base + at[i];
      if (len[i] & PIP_LEN_NARROW) {
        /* the caller's stream is write-only here and far larger than the caches: streaming stores,
         * so that widening the int32 words does not first read the destination lines */
        const int *src = (const int *)(words + off[i]);
#if defined(__x86_64__)
        for (long long k = 0; k < w; k++) _mm_stream_si64((long long *)dst + k, (long long)src[k]);
#else
        for (long long k = 0; k < w; k++) dst[k] = src[k];
#endif
      } else memcpy(dst, words + off[i], sizeof(I) * (size_t)w);
    }
#if defined(__x86_64__)
    _mm_sfence();
#endif
  });
}

/* where a caller buffer lives; managed memory is treated as pageable host memory */
enum MemKind { MEM_PAGEABLE, MEM_PINNED, MEM_DEVICE };
MemKind mem_kind(const void *p, int *device = nullptr)
{
  if (!p) return MEM_PAGEABLE;
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return MEM_PAGEABLE; }
  if (a.type == cudaMemoryTypeDevice) {
    if (device) *device = a.device;
    return MEM_DEVICE;
  }
  return a.type == cudaMemoryTypeHost ? MEM_PINNED : MEM_PAGEABLE;
}
bool is_pinned(const void *p) { return mem_kind(p) == MEM_PINNED; }

/* the calling thread's current device is the caller's: the dense path selects the devices it runs on */
struct KeepCurrentDevice {
  int saved = -1;
  KeepCurrentDevice() { if (cudaGetDevice(&saved) != cudaSuccess) { cudaGetLastError(); saved = -1; } }
  ~KeepCurrentDevice() { if (saved >= 0) cudaSetDevice(saved); }
};

std::mutex g_dense_mu;                  /* one dense call at a time per process (it is parallel inside) */
/* One lane at a time per device and direction on the PCIe link: lanes that all upload, then all solve, then
 * all download move in lockstep and overlap nothing (measured at 8 GPUs: every lane's upload, solve and
 * download each took four times its share and the call took their sum).  With the link handed from lane to
 * lane a chunk goes up at full speed while the previous one is being solved and the one before comes down. */
std::mutex g_h2d_mu[PipEngine::MAX_DEVICES], g_d2h_mu[PipEngine::MAX_DEVICES];
std::vector<int> g_devices;             /* devices a dense call spreads its chunks over (pip_set_devices_dp) */
std::mutex g_devices_mu;

}  // namespace

extern "C" {

/* PIPLIB_B200_CHUNK / PIPLIB_B200_LANES tune the pipeline of the dense path */
static size_t env_size(const char *name, size_t dflt)
{
  const char *v = getenv(name);
  if (!v || !*v) return dflt;
  long long x = atoll(v);
  return x > 0 ? (size_t)x : dflt;
}

int pip_pin_buffer_dp(void *p, size_t bytes)
{
  if (!p || !bytes) return -1;
  if (is_pinned(p)) return 0;
  const cudaError_t e = cudaHostRegister(p, bytes, cudaHostRegisterPortable);
  if (e != cudaSuccess) { cudaGetLastError(); return -1; }
  return 0;
}
void *pip_alloc_pinned_dp(size_t bytes)
{
  void *p = nullptr;
  const cudaError_t e = cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocPortable);
  if (e != cudaSuccess) { cudaGetLastError(); return nullptr; }
  return p;
}
void pip_free_pinned_dp(void *p) { if (p) cudaFreeHost(p); }
int pip_unpin_buffer_dp(void *p)
{
  if (!p) return -1;
  const cudaError_t e = cudaHostUnregister(p);
  if (e != cudaSuccess) { cudaGetLastError(); return -1; }
  return 0;
}
int pip_set_devices_dp(int n, const int *devices)
{
  int count = 0;
  if (cudaGetDeviceCount(&count) != cudaSuccess) { cudaGetLastError(); return -1; }
  std::vector<int> v;
  for (int i = 0; i < n; i++) {
    if (devices[i] < 0 || devices[i] >= count || devices[i] >= PipEngine::MAX_DEVICES) return -1;
    v.push_back(devices[i]);
  }
  std::lock_guard<std::mutex> g(g_devices_mu);
  g_devices = v;                        /* empty: back to the single default device */
  return 0;
}

int pip_solve_dense_dp(long long n, int dom_rows, int dom_cols, const long long *dom,
                       int has_ctx, int ctx_rows, int ctx_cols, const long long *ctx,
                       int bignum, const PipOptions_dp *options,
                       int *status, unsigned long long *hashes,
                       long long *ser, long long ser_cap, long long *ser_off, long long *ser_len)
{
  return pip_solve_dense_info_dp(n, dom_rows, dom_cols, dom, has_ctx, ctx_rows, ctx_cols, ctx, bignum, options,
                                 status, hashes, ser, ser_cap, ser_off, ser_len, nullptr);
}

int pip_solve_dense_info_dp(long long n, int dom_rows, int dom_cols, const long long *dom,
                            int has_ctx, int ctx_rows, int ctx_cols, const long long *ctx,
                            int bignum, const PipOptions_dp *options,
                            int *status, unsigned long long *hashes,
                            long long *ser, long long ser_cap, long long *ser_off, long long *ser_len,
                            PipProblemInfo_dp *info_out)
{
  if (n <= 0) return 0;
  PipInfo *const info = (PipInfo *)info_out;
  std::lock_guard<std::mutex> dense_guard(g_dense_mu);
  KeepCurrentDevice keep_device;
  try {
    const double t0 = wall();
    DenseArgs A = {n, dom_rows, dom_cols, dom, has_ctx, ctx_rows, ctx_cols, ctx, bignum,
                   options ? *options : DEFAULT_OPTIONS};
    /* Caller arrays in device memory: the inputs are converted where they are and the results are written
     * there.  Every device-resident array must be on one device, and the inputs and the outputs each go
     * wholly one way or the other; nothing has been written when such a call is refused. */
    const bool ctx_used = has_ctx && ctx_rows > 0;
    int owner = -1;
    bool other_device = false;
    auto on_device = [&](const void *p) {
      int d = -1;
      if (mem_kind(p, &d) != MEM_DEVICE) return false;
      if (owner >= 0 && d != owner) other_device = true;
      owner = d;
      return true;
    };
    const bool in_device = on_device(dom);
    const bool ctx_device = ctx_used && on_device(ctx);
    int nout = 0, nout_device = 0;
    for (const void *p : {(const void *)status, (const void *)hashes, (const void *)ser, (const void *)ser_off, (const void *)ser_len,
                          (const void *)info})
      if (p) { nout++; nout_device += on_device(p) ? 1 : 0; }
    const bool out_device = nout_device > 0;
    const bool host_decoder = A.opt.Simplify || (A.opt.Compute_dual && !A.opt.Nq);
    if (other_device || (ctx_used && ctx_device != in_device) || (out_device && nout_device != nout) ||
        ((in_device || out_device) && host_decoder))
      return -3;
    std::vector<int> devices;
    {
      std::lock_guard<std::mutex> g(g_devices_mu);
      devices = g_devices;
    }
    if (devices.empty()) devices.push_back(pip_engine_device());
    if (owner >= 0) devices.assign(1, owner);          /* device-resident arrays: the device that owns them */
    const bool keep = ser != nullptr && ser_off != nullptr;
    /* decode on the GPU unless the host-only Simplify post-pass is wanted (PIPLIB_B200_HOST_DECODE=1
     * forces the host decoder, for A/B tests, except for device-resident arrays, which it cannot write) */
    const bool device_decode = !host_decoder && (getenv("PIPLIB_B200_HOST_DECODE") == nullptr || in_device || out_device);
    /* Input stage.  Caller rows in device memory are converted in place (pip_convert_kernel reads them where
     * they are).  Caller buffers in pinned (page-locked) memory are moved by DMA alone: the raw PolyLib rows
     * go up as they are and tab_Matrix2Tableau runs on the device.  Pageable buffers are converted (narrowed
     * to int8 / int32) by the host pool into pinned staging. */
    enum InRoute { IN_HOST_CONVERT, IN_DMA_CONVERT, IN_DEVICE_CONVERT };
    const bool in_pinned = device_decode && is_pinned(dom) && (!ctx_used || is_pinned(ctx)) &&
                           getenv("PIPLIB_B200_HOST_CONVERT") == nullptr;
    const InRoute in_route = in_device ? IN_DEVICE_CONVERT : in_pinned ? IN_DMA_CONVERT : IN_HOST_CONVERT;
    /* Output stage.  Device-resident outputs are written on the device (one device-to-device copy of the
     * chunk's words, pip_emit_device_kernel for the per-problem arrays); a pinned stream receives the words
     * straight from the device; pageable outputs are staged through pinned scratch and widened out of it. */
    enum OutRoute { OUT_STAGED, OUT_PINNED_DMA, OUT_DEVICE };
    const bool out_pinned = device_decode && keep && is_pinned(ser) &&
                            getenv("PIPLIB_B200_STAGED_OUT") == nullptr;
    const OutRoute out_route = out_device ? OUT_DEVICE : out_pinned ? OUT_PINNED_DMA : OUT_STAGED;

    /* chunk schedule: full chunks of CH problems, with a geometric ramp at both ends (CH/8, CH/4,
     * CH/2) so that the GPU starts after one small transfer and the last copy-out is short */
    const size_t CH = env_size("PIPLIB_B200_CHUNK", 1u << 17);
    std::vector<size_t> sizes;
    {
      const size_t ramp = env_size("PIPLIB_B200_RAMP", 3);
      size_t left = (size_t)n;
      std::vector<size_t> head, tail;
      for (size_t k = ramp; k >= 1 && left > 4 * CH * devices.size(); k--) {
        const size_t sz = std::max<size_t>(CH >> k, 1024);
        for (size_t d = 0; d < devices.size(); d++) {
          head.push_back(sz); left -= sz;
          tail.push_back(sz); left -= sz;
        }
      }
      sizes = head;
      while (left > 0) { const size_t sz = std::min(CH, left); sizes.push_back(sz); left -= sz; }
      for (size_t k = tail.size(); k-- > 0;) sizes.push_back(tail[k]);
    }
    const size_t nchunks = sizes.size();
    const size_t lanes = std::max<size_t>(1, std::min<size_t>(std::min<size_t>(env_size("PIPLIB_B200_LANES", 6), PipEngine::MAX_LANES),
                                                              (nchunks + devices.size() - 1) / devices.size()));
    const size_t nworkers = lanes * devices.size();
    const size_t tail_chunks = env_size("PIPLIB_B200_TAIL_CHUNKS", 0) * devices.size();   /* chunks at the end of the call that run with the hand-over (measured: no effect on the call) */
    /* host threads per lane: the lanes' conversion / copy-out phases overlap, so each gets a share */
    const size_t nthreads_default = std::max<size_t>(1, (host_threads() + nworkers - 1) / nworkers);
    std::vector<size_t> firsts(nchunks + 1, 0);
    for (size_t c = 0; c < nchunks; c++) firsts[c + 1] = firsts[c] + sizes[c];
    std::vector<std::string> errors(nworkers);
    std::atomic<long long> cursor(0);
    std::atomic<size_t> next_chunk(0);
    std::atomic<int> width_hint(0);
    std::atomic<int> uniform_hint(getenv("PIPLIB_B200_EXACT_PLAN") ? 0 : 1);
    const bool timing = getenv("PIPLIB_B200_TIMING") != nullptr;
    std::vector<double> tstage(nworkers * 4, 0.0);
    std::vector<PipBatchStats_dp> lane_stats(nworkers);
    for (auto &ls : lane_stats) memset(&ls, 0, sizeof ls);

    /* everything pip_solve derives from the dimensions and the options alone */
    PipConvertShape CS;
    PipDecodeParm uparm;
    int sol_flags0 = 0;
    {
      MatView d0 = {A.dr, A.dc, nullptr, A.dom};
      MatView c0 = {A.cr, A.cc, nullptr, A.ctx};
      const Shape s0 = derive_shape_dims(d0.cols, A.has_ctx ? &c0 : nullptr, A.bignum, A.opt);
      CS.dr = A.dr; CS.dc = A.dc; CS.cr = A.has_ctx ? A.cr : 0; CS.cc = A.cc; CS.has_ctx = A.has_ctx && A.cr > 0;
      CS.Nn = s0.Nn; CS.Np = s0.Np; CS.Bg = s0.Bg; CS.Shift = s0.Shift; CS.Urs = s0.Urs;
      CS.pflags = s0.flags | ((s0.sol_flags == 0 && s0.Urs == 0) ? PIP_F_SIMPLE_SER : 0);
      CS.width = s0.Nn + s0.Np + 1; CS.cwidth = s0.Np + 1;
      uparm.bg = s0.Bg - s0.Nn - 1; uparm.urs = s0.Urs; uparm.flags = s0.sol_flags;
      sol_flags0 = s0.sol_flags;
    }
    (void)sol_flags0;

    /* Mixed input routes (PIPLIB_B200_HOST_LANES=k, default 0): with pinned input, k of the lanes narrow their
     * chunks on the host instead (0.5 KB per problem over the link instead of 4.2 KB) and pull from the same
     * chunk queue.  Measured on a box whose link does 55 GB/s each way: no gain (the upload is not what bounds
     * the call), so it is off; a box with a slower link may want it. */
    size_t host_lanes = 0;
    if (in_route == IN_DMA_CONVERT) {
      if (const char *hv = getenv("PIPLIB_B200_HOST_LANES")) host_lanes = (size_t)std::max(0, atoi(hv));
      host_lanes = std::min<size_t>(host_lanes, lanes > 1 ? lanes - 1 : 0);
    }
    auto worker_main = [&](size_t w) {
      try {
        const int device = devices[w / lanes];
        const InRoute lane_in = (in_route == IN_DMA_CONVERT && (w % lanes) < host_lanes) ? IN_HOST_CONVERT : in_route;
        const size_t nthreads = (in_route == IN_DMA_CONVERT && lane_in == IN_HOST_CONVERT)
                                    ? std::max<size_t>(1, host_threads() / std::max<size_t>(1, host_lanes * devices.size()))
                                    : nthreads_default;
        PipEngine &E = PipEngine::at(device, (int)(w % lanes));
        cudaStream_t s = E.stream();
        pip_cuda_check(cudaSetDevice(device), "cudaSetDevice");
        DenseChunk C;                       /* per-worker scratch, reused from chunk to chunk */
        std::vector<long long> at;
        cudaEvent_t copied = nullptr;
        pip_cuda_check(cudaEventCreateWithFlags(&copied, cudaEventDisableTiming), "cudaEventCreate");
        for (;;) {
          const size_t c = next_chunk.fetch_add(1);          /* chunks go to whichever device / lane is free */
          if (c >= nchunks) break;
          C.first = firsts[c]; C.n = sizes[c];
          const size_t cn = C.n;
          double ta = wall(), tb = ta, tc = ta;
          PipBatchIn in;
          in.n = cn;
          PipProblem uniform;
          struct WidenCtx { PipConvertArgs a; void *pool64; } wc;
          wc.pool64 = nullptr;
          if (lane_in != IN_HOST_CONVERT) {
            /* ---- convert the raw rows on the device: the caller's rows where they are, or a DMA'd copy ---- */
            const size_t dwords = (size_t)A.dr * A.dc, cwords = CS.has_ctx ? (size_t)A.cr * A.cc : 0;
            const pip_i64 *d_dom, *d_ctx;
            if (lane_in == IN_DEVICE_CONVERT) {
              d_dom = A.dom + C.first * dwords;
              d_ctx = cwords ? A.ctx + C.first * cwords : nullptr;
            } else {
              pip_i64 *up_dom = (pip_i64 *)E.device_scratch(0, std::max<size_t>(cn * dwords * 8, 8));
              pip_i64 *up_ctx = (pip_i64 *)E.device_scratch(1, std::max<size_t>(cn * cwords * 8, 8));
              std::lock_guard<std::mutex> link(g_h2d_mu[device]);
              if (dwords) pip_cuda_check(cudaMemcpyAsync(up_dom, A.dom + C.first * dwords, cn * dwords * 8, cudaMemcpyHostToDevice, s), "H2D domain rows");
              if (cwords) pip_cuda_check(cudaMemcpyAsync(up_ctx, A.ctx + C.first * cwords, cn * cwords * 8, cudaMemcpyHostToDevice, s), "H2D context rows");
              pip_cuda_check(cudaEventRecord(copied, s), "cudaEventRecord");
              pip_cuda_check(cudaEventSynchronize(copied), "wait for the upload");      /* (not for the kernels behind it) */
              lane_stats[w].h2d_bytes += cn * (dwords + cwords) * 8;
              d_dom = up_dom; d_ctx = up_ctx;
            }
            const long long stride = 2ll * A.dr * CS.width + 2ll * CS.cr * CS.cwidth;
            void *d_pool = E.device_scratch(2, std::max<size_t>((size_t)cn * stride * 4, 8));
            unsigned char *d_pd = (unsigned char *)E.device_scratch(3, cn * sizeof(PipProblem) + 64);
            int *d_dims = (int *)(d_pd + cn * sizeof(PipProblem));
            int *h_dims = (int *)E.pinned_scratch(0, 64);
            pip_cuda_check(cudaMemsetAsync(d_dims, 0, 16, s), "memset dims");
            PipConvertArgs &ca = wc.a;
            ca.s = CS; ca.dom = d_dom; ca.ctx = d_ctx; ca.n = (long long)cn; ca.stride = stride;
            ca.pool = d_pool; ca.prob = (PipProblem *)d_pd; ca.dims = d_dims;
            pip_cuda_check(pip_launch_convert(&ca, 2, s), "convert kernel");
            pip_cuda_check(cudaMemcpyAsync(h_dims, d_dims, 16, cudaMemcpyDeviceToHost, s), "D2H dims");
            pip_cuda_check(cudaStreamSynchronize(s), "sync after conversion");
            tb = tc = wall();
            uniform.nvar = CS.Nn; uniform.nparm = CS.Np; uniform.ni = h_dims[0]; uniform.nc = h_dims[1];
            uniform.bigparm = CS.Bg; uniform.flags = CS.pflags; uniform.off = 0;
            in.d_prob = (const PipProblem *)d_pd; in.d_pool = d_pool; in.elem_log2 = 2;
            in.uniform = &uniform;
            in.widen_ctx = &wc;
            in.widen_pool = [](void *ctx, cudaStream_t st) -> const void * {
              WidenCtx *w = (WidenCtx *)ctx;
              if (!w->pool64) {
                pip_cuda_check(cudaMalloc(&w->pool64, std::max<size_t>((size_t)w->a.n * w->a.stride * 8, 8)), "cudaMalloc(int64 pool)");
                PipConvertArgs a64 = w->a;
                a64.pool = w->pool64; a64.dims = nullptr;
                pip_cuda_check(pip_launch_convert(&a64, 3, st), "convert kernel (int64)");
              }
              return w->pool64;
            };
          } else {
            /* ---- convert on the host (narrowing) into pinned staging ---- */
            const bool optimistic = uniform_hint.load() != 0;
            if (optimistic) plan_chunk_uniform(A, C); else plan_chunk(A, C, nthreads);
            tb = wall();
            std::atomic<int> mismatch(0);
            void *pool = convert_chunk(A, C, E, nthreads, &width_hint, optimistic ? &mismatch : nullptr);
            bool is_uniform = optimistic;
            if (mismatch.load()) {            /* the number of equality rows varies: exact plan, convert again */
              uniform_hint.store(0);
              plan_chunk(A, C, nthreads);
              pool = convert_chunk(A, C, E, nthreads, &width_hint);
              is_uniform = false;
            }
            tc = wall();
            in.h_prob = C.prob.data(); in.h_pool = pool; in.pool_words = C.pool_elems;
            in.elem_log2 = C.elem_log2;
            if (is_uniform && cn) { uniform = C.prob[0]; uniform.off = 0; in.uniform = &uniform; }
          }
          tstage[w * 4 + 0] += tb - ta; tstage[w * 4 + 1] += tc - tb;
          if (device_decode) {
            in.uniform_decode = &uparm;
            in.stream_out = true;
            /* other lanes keep the machine busy during this chunk's tail -- except at the end of the call */
            in.overlapped = nworkers > 1 && c + tail_chunks < nchunks;
            in.words64 = out_route == OUT_PINNED_DMA || (out_route == OUT_DEVICE && keep);
            in.want_info = info != nullptr;
          }
          double td = wall();
          E.run(in, C.out);
          double te = wall();
          if (wc.pool64) { cudaFree(wc.pool64); wc.pool64 = nullptr; }
          if (device_decode) {
            const PipDeviceOut &D = C.out.dev;
            if (out_route == OUT_DEVICE) {
              /* the chunk's words (one contiguous span of int64) and its per-problem arrays stay on the device */
              long long base = 0;
              if (keep) {
                base = cursor.fetch_add(D.slots);
                if (D.slots && base + D.slots <= ser_cap)
                  pip_cuda_check(cudaMemcpyAsync(ser + base, D.words, (size_t)D.slots * 8, cudaMemcpyDeviceToDevice, s), "D2D quasts");
              }
              pip_cuda_check(pip_launch_emit_device(D.status, D.hash, D.off, D.len, D.info, (long long)cn, base, status + C.first,
                                                    hashes ? hashes + C.first : nullptr,
                                                    keep ? ser_off + C.first : nullptr,
                                                    keep && ser_len ? ser_len + C.first : nullptr,
                                                    info ? info + C.first : nullptr, s), "emit kernel");
              pip_cuda_check(cudaStreamSynchronize(s), "sync after emit");
            } else {
              /* per-problem arrays: SoA on the device -> pinned scratch -> the caller's arrays */
              const size_t soa = cn * (sizeof(int) + sizeof(pip_u64) + 2 * sizeof(long long) + (info ? sizeof(PipInfo) : 0));
              unsigned char *hp = (unsigned char *)E.pinned_scratch(1, soa + 64);
              long long *h_off = (long long *)hp, *h_len = h_off + cn;
              pip_u64 *h_hash = (pip_u64 *)(h_len + cn);
              PipInfo *h_info = (PipInfo *)(h_hash + cn);
              int *h_st = (int *)(h_info + (info ? cn : 0));
              std::unique_lock<std::mutex> link(g_d2h_mu[device]);
              pip_cuda_check(cudaMemcpyAsync(h_off, D.off, cn * 8, cudaMemcpyDeviceToHost, s), "D2H offsets");
              pip_cuda_check(cudaMemcpyAsync(h_len, D.len, cn * 8, cudaMemcpyDeviceToHost, s), "D2H lengths");
              pip_cuda_check(cudaMemcpyAsync(h_hash, D.hash, cn * 8, cudaMemcpyDeviceToHost, s), "D2H hashes");
              if (info) pip_cuda_check(cudaMemcpyAsync(h_info, D.info, cn * sizeof(PipInfo), cudaMemcpyDeviceToHost, s), "D2H reports");
              pip_cuda_check(cudaMemcpyAsync(h_st, D.status, cn * 4, cudaMemcpyDeviceToHost, s), "D2H statuses");
              lane_stats[w].d2h_bytes += soa;
              if (out_route == OUT_PINNED_DMA) {
                /* the chunk's words are one contiguous span of int64: one DMA into the caller's stream */
                const long long total = D.slots;
                const long long base = cursor.fetch_add(total);
                const bool fits = base + total <= ser_cap;
                if (fits && total) {
                  pip_cuda_check(cudaMemcpyAsync(ser + base, D.words, (size_t)total * 8, cudaMemcpyDeviceToHost, s), "D2H quasts");
                  lane_stats[w].d2h_bytes += (size_t)total * 8;
                }
                pip_cuda_check(cudaStreamSynchronize(s), "sync after D2H");
                link.unlock();
                for (size_t i = 0; i < cn; i++) {
                  const int s0 = h_st[i];
                  status[C.first + i] = PIP_STATUS_IS_FINAL(s0) ? s0 : PIP_ST_CAPACITY;
                  ser_off[C.first + i] = base + h_off[i];
                  if (ser_len) ser_len[C.first + i] = h_len[i] & ~PIP_LEN_NARROW;
                }
                if (hashes) memcpy(hashes + C.first, h_hash, cn * 8);
                if (info) memcpy(info + C.first, h_info, cn * sizeof(PipInfo));   /* (not final: all zero already) */
              } else {
                pip_i64 *h_words = nullptr;
                if (keep && D.slots) {
                  h_words = (pip_i64 *)E.pinned_scratch(2, (size_t)D.slots * 8);
                  pip_cuda_check(cudaMemcpyAsync(h_words, D.words, (size_t)D.slots * 8, cudaMemcpyDeviceToHost, s), "D2H quasts");
                  lane_stats[w].d2h_bytes += (size_t)D.slots * 8;
                }
                pip_cuda_check(cudaStreamSynchronize(s), "sync after D2H");
                link.unlock();
                emit_chunk_staged(C.first, cn, h_words, h_st, h_hash, h_off, h_len, status, hashes, ser, ser_cap, ser_off,
                                  ser_len, &cursor, nthreads, at);
                if (info) memcpy(info + C.first, h_info, cn * sizeof(PipInfo));
              }
            }
            PipBatchStats_dp &ls = lane_stats[w];
            ls.pivots += D.stats[0]; ls.cuts += D.stats[1]; ls.subsolves += D.stats[2]; ls.splits += D.stats[3];
            ls.elem_updates += D.stats[4]; ls.cells += D.stats[5]; ls.wrapped += D.stats[8];
            ls.max_rows = std::max(ls.max_rows, (unsigned)D.stats[6]); ls.max_cols = std::max(ls.max_cols, (unsigned)D.stats[7]);
          } else emit_chunk(A, C, status, hashes, ser, ser_cap, ser_off, ser_len, &cursor, nthreads, info);
          tstage[w * 4 + 2] += te - td; tstage[w * 4 + 3] += wall() - te;
          accumulate(lane_stats[w], C.out);
          if (timing)
            fprintf(stderr, "[piplib-b200] chunk %zu device %d lane %zu: rounds %d: %d problems %.3f s | %d problems %.3f s | %d problems %.3f s; d2h %.3f s\n", c, device, w % lanes,
                    C.out.times.rounds, C.out.times.round_n[0], C.out.times.round_s[0], C.out.times.round_n[1], C.out.times.round_s[1],
                    C.out.times.round_n[2], C.out.times.round_s[2], C.out.times.d2h);
          /* the cell chunks are engine-owned and reused by the next run on this lane: drop the views */
          C.out.base.clear();
        }
        cudaEventDestroy(copied);
      } catch (const std::exception &e) { errors[w] = e.what(); }
    };
    if (nworkers <= 1) worker_main(0);
    else {
      std::vector<std::thread> th;
      for (size_t l = 0; l < nworkers; l++) th.emplace_back(worker_main, l);
      for (auto &x : th) x.join();
    }
    for (const std::string &e : errors) if (!e.empty()) throw std::runtime_error(e);
    const long long total = cursor.load();
    if (ser_off && out_route == OUT_DEVICE) {
      pip_cuda_check(cudaSetDevice(owner), "cudaSetDevice");
      pip_cuda_check(cudaMemcpy(ser_off + n, &total, sizeof total, cudaMemcpyHostToDevice), "H2D words used");
    } else if (ser_off) ser_off[n] = total;
    if (timing) {
      static const char *const in_name[] = {"pageable: host conversion", "pinned: DMA + device conversion", "device: conversion in place"};
      static const char *const out_name[] = {"pageable: staged", "pinned: DMA", "device: written in place"};
      for (size_t l = 0; l < nworkers; l++)
        fprintf(stderr, "[piplib-b200] device %d lane %zu: plan %.3f convert %.3f run %.3f emit %.3f s\n", devices[l / lanes], l % lanes,
                tstage[l * 4], tstage[l * 4 + 1], tstage[l * 4 + 2], tstage[l * 4 + 3]);
      fprintf(stderr, "[piplib-b200] total %.3f s, %zu chunks, %zu devices x %zu lanes (%zu of them convert on the host), pool %u, input %s, output %s\n",
              wall() - t0, nchunks, devices.size(), lanes, in_route == IN_DMA_CONVERT ? host_lanes : in_route == IN_HOST_CONVERT ? lanes : 0,
              host_threads(), in_name[in_route], out_name[out_route]);
    }
    PipBatchStats_dp acc;
    memset(&acc, 0, sizeof acc);
    for (size_t l = 0; l < nworkers; l++) merge_stats(acc, lane_stats[l]);
    acc.seconds_host = (wall() - t0) - acc.seconds_h2d - acc.seconds_kernel - acc.seconds_d2h;
    publish_stats(acc);
    if (keep && total > ser_cap) return -2;
  } catch (const std::exception &e) {
    fprintf(stderr, "%s\n", e.what());
    return -1;
  }
  return 0;
}

struct pip_device_batch {
  DenseArgs A;
  DenseChunk C;
  PipProblem *d_prob = nullptr;
  void *d_pool = nullptr;
  bool fetched = false;
  bool device_decode = false;           /* run() = solve + decode on the device (serialised quasts stay in HBM) */
  bool uniform = false;
  bool keep_info = false;               /* runs write the per-problem reports (pip_device_batch_info(b, NULL)) */
  PipProblem shape;
  std::vector<PipDecodeParm> parm;
  int device = 0;
  /* a big device job runs as a few parts of falling size on engine lanes of their own (pip_device_batch_run) */
  struct Part { size_t first = 0, n = 0; PipBatchOut out; std::string error; };
  std::vector<Part> parts;
  cudaStream_t clock_stream = nullptr;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
};

pip_device_batch *pip_device_batch_create(long long n, int dom_rows, int dom_cols, const long long *dom,
                                          int has_ctx, int ctx_rows, int ctx_cols, const long long *ctx,
                                          int bignum, const PipOptions_dp *options)
{
  try {
    pip_device_batch *b = new pip_device_batch;
    b->A = {n, dom_rows, dom_cols, dom, has_ctx, ctx_rows, ctx_cols, ctx, bignum, options ? *options : DEFAULT_OPTIONS};
    b->C.first = 0; b->C.n = (size_t)n;
    const size_t nthreads = host_threads();
    plan_chunk(b->A, b->C, nthreads);
    PipEngine &E = PipEngine::get();
    b->device = E.device_id();
    void *pool = convert_chunk(b->A, b->C, E, nthreads, nullptr);
    pip_cuda_check(cudaMalloc((void **)&b->d_prob, sizeof(PipProblem) * (size_t)n), "cudaMalloc(problems)");
    pip_cuda_check(cudaMalloc(&b->d_pool, (b->C.pool_elems + 8) << b->C.elem_log2), "cudaMalloc(pool)");
    pip_cuda_check(cudaMemcpy(b->d_prob, b->C.prob.data(), sizeof(PipProblem) * (size_t)n, cudaMemcpyHostToDevice), "H2D problems");
    pip_cuda_check(cudaMemcpy(b->d_pool, pool, b->C.pool_elems << b->C.elem_log2, cudaMemcpyHostToDevice), "H2D pool");
    /* the device job = solve + decode unless the decode needs the host (Simplify, dual with equalities) */
    b->device_decode = !b->A.opt.Simplify && !(b->A.opt.Compute_dual && !b->A.opt.Nq) &&
                       getenv("PIPLIB_B200_HOST_DECODE") == nullptr;
    b->uniform = n > 0;
    b->parm.resize((size_t)n);
    for (size_t i = 0; i < (size_t)n; i++) {
      const Shape &sh = b->C.shapes[i];
      b->parm[i].bg = sh.Bg - sh.Nn - 1; b->parm[i].urs = sh.Urs; b->parm[i].flags = sh.sol_flags;
      if (sh.Nl != b->C.shapes[0].Nl || sh.Nm != b->C.shapes[0].Nm) b->uniform = false;
    }
    if (b->uniform) { b->shape = b->C.prob[0]; b->shape.off = 0; }
    b->A.dom = nullptr; b->A.ctx = nullptr;          /* the caller's arrays are not kept */
    return b;
  } catch (const std::exception &e) {
    fprintf(stderr, "%s\n", e.what());
    return nullptr;
  }
}

/* fetch_cells = 0: the whole device job with the results left in HBM -- solve, then decode to serialised
 * quasts (the same kernels the host-buffer path runs); fetch_cells = 1: solve + cell gather, cells copied
 * to the host (host decoder) */
int pip_device_batch_run(pip_device_batch *b, int fetch_cells, float *device_ms)
{
  try {
    PipBatchIn in;
    in.n = b->C.n; in.h_prob = b->C.prob.data();
    in.d_prob = b->d_prob; in.d_pool = b->d_pool; in.elem_log2 = b->C.elem_log2;
    if (b->uniform) in.uniform = &b->shape;
    const bool stream = !fetch_cells && b->device_decode;
    if (stream) {
      if (b->uniform) in.uniform_decode = &b->parm[0]; else in.h_decode = b->parm.data();
      in.stream_out = true;
      in.want_info = b->keep_info;
    } else in.fetch_cells = fetch_cells != 0;
    b->parts.clear();
    /* A launch ends with its heaviest problems, one warp each, on an idle machine (loop nests: the last ~12 ms
     * of 128 at 10^6 problems; DESIGN.md section 6).  So a big job runs as parts of falling size on engine lanes
     * of their own, launched in that order: the tail of a part is filled by the CTAs of the next one, and the
     * last part is small enough for the heavy-problem hand-over.  The results of every part stay in its lane's
     * buffers in HBM.  Measured at 10^6 problems (profiles/r2_device_job_parts.log): 129 -> 124.4 ms with 3 or 4
     * parts, 127.5 with 6 or 8; which part holds the largest trees moves it by a few ms.
     * PIPLIB_B200_DEVICE_PARTS=1 runs the job as one launch */
    size_t nparts = 1;
    if (stream && b->C.n > ((size_t)1 << 19)) nparts = std::min<size_t>(env_size("PIPLIB_B200_DEVICE_PARTS", 3), PipEngine::MAX_LANES);
    if (nparts > 1) {
      double share[8] = {0.55, 0.30, 0.15, 0.08, 0.04, 0.02, 0.01, 0.005};
      if (const char *sv = getenv("PIPLIB_B200_DEVICE_SHARES")) {       /* "0.6,0.3,0.1": tuning */
        nparts = 0;
        for (const char *c = sv; *c && nparts < 8;) {
          char *end = nullptr;
          share[nparts++] = strtod(c, &end);
          c = (*end == ',') ? end + 1 : end;
          if (end == c && *end != ',') break;
        }
        if (nparts < 1) nparts = 1;
      }
      double sum = 0;
      for (size_t q = 0; q < nparts; q++) sum += share[q];
      b->parts.resize(nparts);
      size_t at = 0;
      for (size_t q = 0; q < nparts; q++) {
        size_t cnt = q + 1 == nparts ? b->C.n - at : (size_t)((double)b->C.n * share[q] / sum) & ~(size_t)1023;
        b->parts[q].first = at; b->parts[q].n = cnt;
        at += cnt;
      }
      pip_cuda_check(cudaSetDevice(b->device), "cudaSetDevice");
      if (!b->clock_stream) {
        pip_cuda_check(cudaStreamCreateWithFlags(&b->clock_stream, cudaStreamNonBlocking), "cudaStreamCreate");
        pip_cuda_check(cudaEventCreate(&b->ev0), "cudaEventCreate");
        pip_cuda_check(cudaEventCreate(&b->ev1), "cudaEventCreate");
      }
      pip_cuda_check(cudaEventRecord(b->ev0, b->clock_stream), "cudaEventRecord");
      std::atomic<int> turn(0);            /* parts enter their engines in order of size */
      auto part_main = [&](size_t q) {
        pip_device_batch::Part &P = b->parts[q];
        try {
          PipBatchIn pin = in;
          pin.n = P.n; pin.h_prob = b->C.prob.data() + P.first; pin.d_prob = b->d_prob + P.first;
          if (pin.h_decode) pin.h_decode = b->parm.data() + P.first;
          pin.overlapped = q + 1 < b->parts.size();
          /* part q enters its engine 400 us after part q - 1 did (its launches are queued behind) */
          while (turn.load() < (int)q) std::this_thread::yield();
          if (q) std::this_thread::sleep_for(std::chrono::microseconds(400));
          turn.store((int)q + 1);
          PipEngine::at(b->device, (int)q).run(pin, P.out);
        } catch (const std::exception &e) {
          P.error = e.what();
          if (turn.load() <= (int)q) turn.store((int)q + 1);
        }
      };
      std::vector<std::thread> th;
      for (size_t q = 1; q < nparts; q++) th.emplace_back(part_main, q);
      part_main(0);
      for (auto &t : th) t.join();
      pip_cuda_check(cudaEventRecord(b->ev1, b->clock_stream), "cudaEventRecord");
      pip_cuda_check(cudaEventSynchronize(b->ev1), "cudaEventSynchronize");
      for (auto &P : b->parts) if (!P.error.empty()) throw std::runtime_error(P.error);
      float ms = 0;
      pip_cuda_check(cudaEventElapsedTime(&ms, b->ev0, b->ev1), "cudaEventElapsedTime");
      b->fetched = false;
      if (device_ms) *device_ms = ms;
      PipBatchStats_dp st;
      memset(&st, 0, sizeof st);
      for (auto &P : b->parts) {
        const PipDeviceOut &D = P.out.dev;
        st.pivots += D.stats[0]; st.cuts += D.stats[1]; st.subsolves += D.stats[2]; st.splits += D.stats[3];
        st.elem_updates += D.stats[4]; st.cells += D.stats[5];
        st.max_rows = std::max(st.max_rows, (unsigned)D.stats[6]); st.max_cols = std::max(st.max_cols, (unsigned)D.stats[7]);
        st.wrapped += D.stats[8];
        accumulate(st, P.out);
      }
      st.device_ms = ms;
      publish_stats(st);
      return 0;
    }
    PipEngine &E = PipEngine::at(b->device, 0);
    E.run(in, b->C.out);
    b->fetched = fetch_cells != 0;
    if (device_ms) *device_ms = b->C.out.times.device_ms;
    if (stream) {
      PipBatchStats_dp st;
      memset(&st, 0, sizeof st);
      const PipDeviceOut &D = b->C.out.dev;
      st.pivots = D.stats[0]; st.cuts = D.stats[1]; st.subsolves = D.stats[2]; st.splits = D.stats[3];
      st.elem_updates = D.stats[4]; st.cells = D.stats[5]; st.max_rows = (unsigned)D.stats[6]; st.max_cols = (unsigned)D.stats[7];
      st.wrapped = D.stats[8];
      accumulate(st, b->C.out);
      publish_stats(st);
    } else account(b->C.out, 0);
  } catch (const std::exception &e) {
    fprintf(stderr, "%s\n", e.what());
    return -1;
  }
  return 0;
}

int pip_device_batch_results(pip_device_batch *b, int *status, unsigned long long *hashes)
{
  if (!b->parts.empty()) {               /* last run went in parts: every lane holds its part's arrays */
    try {
      pip_cuda_check(cudaSetDevice(b->device), "cudaSetDevice");
      for (auto &P : b->parts) {
        const PipDeviceOut &D = P.out.dev;
        pip_cuda_check(cudaMemcpy(status + P.first, D.status, P.n * sizeof(int), cudaMemcpyDeviceToHost), "D2H statuses");
        if (hashes) pip_cuda_check(cudaMemcpy(hashes + P.first, D.hash, P.n * sizeof(pip_u64), cudaMemcpyDeviceToHost), "D2H hashes");
      }
      for (size_t i = 0; i < b->C.n; i++) if (!PIP_STATUS_IS_FINAL(status[i])) status[i] = PIP_ST_CAPACITY;
    } catch (const std::exception &e) {
      fprintf(stderr, "%s\n", e.what());
      return -1;
    }
    return 0;
  }
  const PipDeviceOut &D = b->C.out.dev;
  if (D.status) {                        /* last run decoded on the device: statuses and hashes are in HBM */
    try {
      pip_cuda_check(cudaSetDevice(b->device), "cudaSetDevice");
      pip_cuda_check(cudaMemcpy(status, D.status, b->C.n * sizeof(int), cudaMemcpyDeviceToHost), "D2H statuses");
      for (size_t i = 0; i < b->C.n; i++) if (!PIP_STATUS_IS_FINAL(status[i])) status[i] = PIP_ST_CAPACITY;
      if (hashes) pip_cuda_check(cudaMemcpy(hashes, D.hash, b->C.n * sizeof(pip_u64), cudaMemcpyDeviceToHost), "D2H hashes");
    } catch (const std::exception &e) {
      fprintf(stderr, "%s\n", e.what());
      return -1;
    }
    return 0;
  }
  if (b->C.out.res.size() != b->C.n) return -1;
  if (hashes && !b->fetched) return -3;
  if (hashes) emit_chunk(b->A, b->C, status, hashes, nullptr, 0, nullptr, nullptr, nullptr, host_threads());
  else for (size_t i = 0; i < b->C.n; i++) status[i] = b->C.out.res[i].status;
  return 0;
}

int pip_device_batch_info(pip_device_batch *b, PipProblemInfo_dp *info_out)
{
  PipInfo *const info = (PipInfo *)info_out;
  if (!info) { b->keep_info = true; return 0; }
  try {
    if (!b->parts.empty()) {             /* last run went in parts: every lane holds its part's reports */
      for (auto &P : b->parts) if (!P.out.dev.info) return -3;
      pip_cuda_check(cudaSetDevice(b->device), "cudaSetDevice");
      for (auto &P : b->parts)
        pip_cuda_check(cudaMemcpy(info + P.first, P.out.dev.info, P.n * sizeof(PipInfo), cudaMemcpyDeviceToHost), "D2H reports");
      return 0;
    }
    const PipDeviceOut &D = b->C.out.dev;
    if (D.status) {                      /* last run decoded on the device */
      if (!D.info) return -3;
      pip_cuda_check(cudaSetDevice(b->device), "cudaSetDevice");
      pip_cuda_check(cudaMemcpy(info, D.info, b->C.n * sizeof(PipInfo), cudaMemcpyDeviceToHost), "D2H reports");
      return 0;
    }
    if (b->C.out.res.size() != b->C.n) return -1;
    for (size_t i = 0; i < b->C.n; i++) info[i] = pip_info_of(b->C.out.res[i]);
  } catch (const std::exception &e) {
    fprintf(stderr, "%s\n", e.what());
    return -1;
  }
  return 0;
}

void pip_device_batch_destroy(pip_device_batch *b)
{
  if (!b) return;
  cudaFree(b->d_prob); cudaFree(b->d_pool);
  if (b->ev0) cudaEventDestroy(b->ev0);
  if (b->ev1) cudaEventDestroy(b->ev1);
  if (b->clock_stream) cudaStreamDestroy(b->clock_stream);
  delete b;
}

}  // extern "C"
