/* Host-side batch engine (see pip_engine.h).  Plain CUDA runtime; no torch, no CPU solver. */
#include "pip_engine.h"

#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <mutex>
#include <stdexcept>
#include <string>

#include "../../include/piplib_b200.h"
#include "pip_kernels.h"

void pip_cuda_check(cudaError_t e, const char *what)
{
  if (e != cudaSuccess)
    throw std::runtime_error(std::string("piplib-b200: CUDA error in ") + what + ": " + cudaGetErrorString(e));
}
#define CK(x) pip_cuda_check((x), #x)

namespace {

double now_s()
{
  return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

struct DevBuf {
  void *p = nullptr;
  size_t cap = 0;
  void reserve(size_t bytes)
  {
    if (bytes <= cap) return;
    if (p) CK(cudaFree(p));
    p = nullptr; cap = 0;
    size_t want = bytes + bytes / 8 + 256;
    CK(cudaMalloc(&p, want));
    cap = want;
  }
  void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
};
struct PinBuf {
  void *p = nullptr;
  size_t cap = 0;
  void reserve(size_t bytes)
  {
    if (bytes <= cap) return;
    if (p) CK(cudaFreeHost(p));
    p = nullptr; cap = 0;
    size_t want = bytes + bytes / 8 + 256;
    CK(cudaHostAlloc(&p, want, cudaHostAllocDefault));
    cap = want;
  }
};

/* the size-class ladder */
/* team = 0: `warps` warps, one problem each; team = t: `warps` CTAs of t warps, one problem per CTA (class M) */
struct ClassSpec { int level; int shared; long long words; int warps; int warps_per_cta; long long stack_words; int team; };
const long long S_MAX_WORDS = 3328;          /* 26 KB: at least 8 warps of class S per SM */
#ifndef PIP_S32_WIDE_MAX_WORDS
#define PIP_S32_WIDE_MAX_WORDS 1700          /* 13.3 KB: 16 warps of class S32 per SM stay resident */
#endif
const long long S32_WIDE_MAX_WORDS = PIP_S32_WIDE_MAX_WORDS;
const ClassSpec G_LADDER[] = {
    {3, 0, 1ll << 15, 148 * 8, 4, 1ll << 17, 0},
    {4, 0, 1ll << 17, 148 * 4, 4, 1ll << 19, 4},
    {5, 0, 1ll << 19, 148 * 2, 2, 1ll << 21, 8},
    {6, 0, 1ll << 22, 148, 1, 1ll << 23, 16},
    {7, 0, 1ll << 24, 32, 1, 1ll << 25, 16},
    {8, 0, 1ll << 26, 8, 1, 1ll << 27, 16},
};
const int N_G = sizeof(G_LADDER) / sizeof(G_LADDER[0]);

}  // namespace

static std::atomic<int> g_device(0);
static std::atomic<int> g_donation(-1);      /* subtree donation: -1 automatic, 0 off, 1 on (pip_set_donation_dp) */
void pip_engine_set_donation(int mode) { g_donation = mode; }
/* the device the calling thread works on: the engine's own device while one of its runs is in progress
 * (the whole-grid class is entered from inside PipEngine::run), else the default of pip_set_device_dp */
static thread_local int t_run_device = -1;
int pip_engine_device() { return t_run_device >= 0 ? t_run_device : g_device.load(); }

struct PipEngine::Impl {
  std::mutex mu;
  int device = -1, sm_count = 0;
  size_t smem_optin = 0;
  bool inited = false;
  cudaStream_t stream = nullptr;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  DevBuf d_prob, d_pool, d_res, d_cells, d_stack, d_gwork, d_queue, d_order, d_off, d_compact, d_total, d_prof, d_parm, d_hash;
  DevBuf d_so_status, d_so_hash, d_so_off, d_so_len, d_so_ctl;     /* stream_out: per-problem arrays, control + stats */
  DevBuf d_so_info;                /* stream_out: per-problem reports, when asked for */
  DevBuf d_image;                  /* arena images of a uniform batch (pip_image_kernel) */
  DevBuf d_stl_offers, d_stl_segs, d_stl_next, d_stl_hwm, d_stl_head_next, d_stl_head_hwm, d_stl_ctl;   /* subtree donation */
  DevBuf d_heavy;                /* problems handed over to the donation launch */
  DevBuf d_scratch[4];
  PinBuf h_scratch[4];
  PinBuf h_hash;
  PinBuf h_res, h_total, h_input, h_ctl;
  std::vector<PinBuf> h_chunks;     /* one per round, reused across calls */

  void init()
  {
    if (inited) return;
    if (device < 0) device = g_device.load();
    CK(cudaSetDevice(device));
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10)
      throw std::runtime_error("piplib-b200: this library is built for sm_100a (B200) only; device is sm_" +
                               std::to_string(prop.major) + std::to_string(prop.minor));
    sm_count = prop.multiProcessorCount;
    smem_optin = prop.sharedMemPerBlockOptin;
    CK(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
    CK(cudaEventCreate(&ev0));
    CK(cudaEventCreate(&ev1));
    inited = true;
  }
};

PipEngine::PipEngine() : impl_(new Impl) {}
PipEngine &PipEngine::at(int device, int i)
{
  /* engines are created on first use and live for the process: [device][lane] */
  static std::mutex mu;
  static PipEngine *table[MAX_DEVICES][MAX_LANES] = {{nullptr}};
  if (device < 0 || device >= MAX_DEVICES) throw std::runtime_error("piplib-b200: device index out of range");
  if (i < 0) i = 0;
  i %= MAX_LANES;
  std::lock_guard<std::mutex> g(mu);
  if (!table[device][i]) { table[device][i] = new PipEngine; table[device][i]->impl_->device = device; }
  return *table[device][i];
}
PipEngine &PipEngine::lane(int i) { return at(g_device.load(), i); }
int PipEngine::set_device(int dev)
{
  if (dev < 0 || dev >= MAX_DEVICES) return -1;
  g_device = dev;          /* engines are per device: the default only selects which set serves the next call */
  return 0;
}
int PipEngine::device_id() { return impl_->device; }
void *PipEngine::pinned_input(size_t bytes)
{
  Impl &E = *impl_;
  std::lock_guard<std::mutex> g(E.mu);
  E.init();
  CK(cudaSetDevice(E.device));
  E.h_input.reserve(bytes);
  return E.h_input.p;
}
void *PipEngine::device_scratch(int which, size_t bytes)
{
  Impl &E = *impl_;
  std::lock_guard<std::mutex> g(E.mu);
  E.init();
  CK(cudaSetDevice(E.device));
  E.d_scratch[which & 3].reserve(bytes);
  return E.d_scratch[which & 3].p;
}
void *PipEngine::pinned_scratch(int which, size_t bytes)
{
  Impl &E = *impl_;
  std::lock_guard<std::mutex> g(E.mu);
  E.init();
  CK(cudaSetDevice(E.device));
  E.h_scratch[which & 3].reserve(bytes);
  return E.h_scratch[which & 3].p;
}
int PipEngine::sm_count() { std::lock_guard<std::mutex> g(impl_->mu); impl_->init(); return impl_->sm_count; }
cudaStream_t PipEngine::stream() { std::lock_guard<std::mutex> g(impl_->mu); impl_->init(); return impl_->stream; }

/* Top of the ladder for non-parametric problems: the few that are still open when the classes with
 * thousands of cut rows are reached get the whole grid, one after the other (class L, pip_large.h),
 * instead of one CTA each with the other SMs idle.  Writes the record and the cells of problem
 * order[q] where warp q of a team round would have put them. */
#ifndef PIP_LARGE_FROM_DEFAULT
#define PIP_LARGE_FROM_DEFAULT 3      /* measured: vivien32-shaped batch 5.44 -> 3.90 s (its last 2 problems 2.87 -> 1.31 s) */
#endif
static bool large_eligible(const PipProblem &P)
{
  return P.nparm == 0 && P.nc == 0 && P.bigparm < 0 && !(P.flags & (PIP_F_DUAL | PIP_F_DEEPEST));
}

static void run_large_round(const PipBatchIn &in, const PipProblem *h_prob, const void *d_pool, int elem_log2,
                            const std::vector<int> &order, PipCell *d_cells,
                            long long per_warp, PipResult *d_res, cudaStream_t s)
{
  std::vector<long long> tab;
  std::vector<unsigned char> raw;
  std::vector<PipCell_dp> cells((size_t)in.sol_size + 8);
  for (size_t q = 0; q < order.size(); q++) {
    const int i = order[q];
    const PipProblem &P = h_prob[i];
    const int ncol = P.nvar + 1;
    tab.resize((size_t)P.ni * ncol);
    /* the problem's words: from the host pool, or (device-resident batches) fetched from the device pool */
    const size_t esz = (size_t)1 << elem_log2;
    const unsigned char *src = (in.h_pool && elem_log2 == in.elem_log2) ? (const unsigned char *)in.h_pool + (size_t)P.off * esz : nullptr;
    if (!src) {
      raw.resize(tab.size() * esz);
      CK(cudaMemcpyAsync(raw.data(), (const unsigned char *)d_pool + (size_t)P.off * esz, raw.size(), cudaMemcpyDeviceToHost, s));
      CK(cudaStreamSynchronize(s));
      src = raw.data();
    }
    for (size_t w = 0; w < tab.size(); w++)
      tab[w] = elem_log2 == 0 ? (long long)((const signed char *)src)[w]
             : elem_log2 == 2 ? (long long)((const int *)src)[w] : ((const long long *)src)[w];
    PipResult r;
    memset(&r, 0, sizeof r);
    r.status = PIP_ST_CAPACITY;
    r.cell_off = (pip_i64)q * per_warp;
    pip_large_problem *lp = pip_large_create_dp(P.nvar, P.ni, (P.flags & PIP_F_INT) ? 1 : 0, tab.data(), 1 << 16,
                                                in.sol_size, in.maxcol);
    if (!lp) throw std::runtime_error("piplib-b200: large-tableau class: allocation failed");
    int st = 0, nc = 0;
    long long info[12] = {0};
    const bool ok = pip_large_run_dp(lp, nullptr) == 0 &&
                    pip_large_fetch_dp(lp, &st, cells.data(), (int)cells.size(), &nc, info) == 0;
    pip_large_destroy_dp(lp);
    if (!ok) throw std::runtime_error("piplib-b200: large-tableau class: launch failed");
    r.status = st;
    r.ncells = st == PIP_ST_OK ? nc : 0;
    r.pivots = (unsigned)info[0]; r.cuts = (unsigned)info[1];
    r.max_rows = (unsigned)(P.nvar + info[3]); r.max_cols = (unsigned)ncol;
    bool wide = false;
    for (int c = 0; c < r.ncells; c++) wide = wide || !PIP_CELL_FITS(cells[c].p1, cells[c].p2);
    r.rflags = wide ? PIP_RES_WIDE : 0u;
    if (r.ncells) CK(cudaMemcpyAsync(d_cells + r.cell_off, cells.data(), sizeof(PipCell) * (size_t)r.ncells, cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync(d_res + i, &r, sizeof r, cudaMemcpyHostToDevice, s));
    CK(cudaStreamSynchronize(s));        /* cells / r are reused by the next problem */
  }
}

namespace {
struct RunDeviceScope {          /* pip_engine_device() answers with this engine's device while it runs */
  int saved;
  explicit RunDeviceScope(int d) : saved(t_run_device) { t_run_device = d; }
  ~RunDeviceScope() { t_run_device = saved; }
};
}  // namespace

void PipEngine::run(const PipBatchIn &in, PipBatchOut &out)
{
  Impl &E = *impl_;
  std::lock_guard<std::mutex> g(E.mu);
  E.init();
  CK(cudaSetDevice(E.device));
  RunDeviceScope scope(E.device);
  const size_t n = in.n;
  const bool stream_out = in.stream_out;
  const bool ser_mode = in.h_decode != nullptr || in.uniform_decode != nullptr;
  if (stream_out && !ser_mode) throw std::runtime_error("piplib-b200: stream_out needs the device decoder");
  if (!in.h_prob && !(in.uniform && in.d_prob)) throw std::runtime_error("piplib-b200: batch without descriptors");
  if (stream_out) { out.res.clear(); out.base.clear(); out.hashes.clear(); }
  else { out.res.assign(n, PipResult()); out.base.assign(n, nullptr); }
  out.times = PipBatchTimes();
  out.dev = PipDeviceOut();
  if (n == 0) return;
  const double t_begin = now_s();
  cudaStream_t s = E.stream;

  /* ---- inputs ------------------------------------------------------------------------- */
  const PipProblem *d_prob = in.d_prob;
  const void *d_pool = in.d_pool;
  int elem_log2 = in.elem_log2;
  double t0 = now_s();
  if (!d_prob) {
    E.d_prob.reserve(n * sizeof(PipProblem));
    CK(cudaMemcpyAsync(E.d_prob.p, in.h_prob, n * sizeof(PipProblem), cudaMemcpyHostToDevice, s));
    d_prob = (const PipProblem *)E.d_prob.p;
    out.times.h2d_bytes += n * sizeof(PipProblem);
  }
  if (!d_pool) {
    const size_t pool_bytes = in.pool_words << in.elem_log2;
    E.d_pool.reserve(std::max<size_t>(pool_bytes, 8));
    CK(cudaMemcpyAsync(E.d_pool.p, in.h_pool, pool_bytes, cudaMemcpyHostToDevice, s));
    d_pool = E.d_pool.p;
    out.times.h2d_bytes += pool_bytes;
  }
  /* per-problem records start as PENDING (written on the device: nothing to upload) */
  E.d_res.reserve(n * sizeof(PipResult));
  CK(pip_launch_init_results((PipResult *)E.d_res.p, (long long)n, s));
  PipResult *h_res = nullptr;            /* host mirror, fetched only when some problem has to change class */
  auto need_h_res = [&]() {
    if (h_res) return;
    E.h_res.reserve(n * sizeof(PipResult));
    h_res = (PipResult *)E.h_res.p;
  };
  if (in.h_decode) {
    E.d_parm.reserve(n * sizeof(PipDecodeParm));
    CK(cudaMemcpyAsync(E.d_parm.p, in.h_decode, n * sizeof(PipDecodeParm), cudaMemcpyHostToDevice, s));
    out.times.h2d_bytes += n * sizeof(PipDecodeParm);
  }
  const PipDecodeParm *d_parm = in.h_decode ? (const PipDecodeParm *)E.d_parm.p : nullptr;
  if (ser_mode && !stream_out) {
    E.d_hash.reserve(n * sizeof(pip_u64));
    CK(cudaMemsetAsync(E.d_hash.p, 0, n * sizeof(pip_u64), s));
  }
  PipStreamOut so;
  memset(&so, 0, sizeof so);
  long long slots_done = 0;              /* stream_out: slots reserved by the rounds completed so far */
  unsigned long long stats_prev[PIP_SO_NSTAT] = {0};   /* ... and the device counters at the end of the last good round */
  unsigned long long *h_ctl = nullptr;
  if (stream_out) {
    E.d_so_status.reserve(n * sizeof(int));
    E.d_so_hash.reserve(n * sizeof(pip_u64));
    E.d_so_off.reserve(n * sizeof(long long));
    E.d_so_len.reserve(n * sizeof(long long));
    E.d_so_ctl.reserve((PIP_SO_NCTL + PIP_SO_NSTAT) * sizeof(unsigned long long));
    CK(cudaMemsetAsync(E.d_so_ctl.p, 0, (PIP_SO_NCTL + PIP_SO_NSTAT) * sizeof(unsigned long long), s));
    E.h_ctl.reserve((PIP_SO_NCTL + PIP_SO_NSTAT) * sizeof(unsigned long long));
    h_ctl = (unsigned long long *)E.h_ctl.p;
    const long long hint = in.words_hint > 0 ? in.words_hint : (long long)n * (in.words64 ? 640 : 384);
    E.d_compact.reserve((size_t)std::max<long long>(hint, 1024) * sizeof(pip_u64));
    so.ctl = (unsigned long long *)E.d_so_ctl.p;
    so.stats = so.ctl + PIP_SO_NCTL;
    so.cap = (long long)(E.d_compact.cap / sizeof(pip_u64));
    so.words64 = in.words64 ? 1 : 0;
    so.status = (int *)E.d_so_status.p; so.hash = (pip_u64 *)E.d_so_hash.p;
    so.off = (long long *)E.d_so_off.p; so.len = (long long *)E.d_so_len.p;
    if (in.want_info) {
      /* every problem's report is written by the decode pass of each round it takes part in (the last one wins) */
      E.d_so_info.reserve(n * sizeof(PipInfo));
      CK(cudaMemsetAsync(E.d_so_info.p, 0, n * sizeof(PipInfo), s));
      so.info = (PipInfo *)E.d_so_info.p;
    }
  }
  E.d_queue.reserve(64);
  E.d_prof.reserve(sizeof(unsigned long long) * PIP_NPHASE);
  CK(cudaMemsetAsync(E.d_prof.p, 0, sizeof(unsigned long long) * PIP_NPHASE, s));
  E.d_total.reserve(64);
  E.h_total.reserve(64);
  out.times.h2d = now_s() - t0;          /* enqueue time only: the copies overlap what follows on the stream */

  /* ---- plan: class S32 (int32 storage, shared memory) for problems shipped with narrow inputs,
   * class S (int64, shared memory) for everything else whose level-2 working set fits an arena,
   * the global-memory ladder for the rest.  A uniform batch is planned once from its shape. */
  const bool try32 = in.elem_log2 <= 2 && getenv("PIPLIB_B200_NO_INT32") == nullptr;
  std::vector<int> cls(n);              /* -2 = class S32, -1 = class S, k = G_LADDER[k] */
  long long s_words = 0, s32_words = 0, s32_wide_words = 0, est_cells_total = 0;
  bool all_sized = true;
  auto plan_one = [&](const PipProblem &P) -> int {
    if (!(P.flags & PIP_F_SIMPLE_SER)) all_sized = false;
    int c;
    long long w = pip_layout_words(P.nvar, P.nparm, P.ni, P.nc, P.flags, 2, 8);
    if (w <= S_MAX_WORDS && !(P.flags & (PIP_F_DUAL | PIP_F_DEEPEST))) {   /* options: global-memory classes only */
      c = try32 ? -2 : -1;
      s_words = std::max(s_words, w);
      if (try32) {
        s32_words = std::max(s32_words, pip_layout_words(P.nvar, P.nparm, P.ni, P.nc, P.flags, 2, 4));
        s32_wide_words = std::max(s32_wide_words, pip_layout_words(P.nvar, P.nparm, P.ni, P.nc, P.flags, PIP_LEVEL_S_WIDE, 4));
      }
    } else {
      int k = 0;
      while (k < N_G - 1 && pip_layout_words(P.nvar, P.nparm, P.ni, P.nc, P.flags, G_LADDER[k].level, 8) > G_LADDER[k].words) k++;
      c = k;
    }
    return c;
  };
  if (in.uniform) {
    const int c = plan_one(*in.uniform);
    std::fill(cls.begin(), cls.end(), c);
    est_cells_total = (long long)n * (3ll * (1 + in.uniform->nvar * (2 + in.uniform->nparm)) + 32);
  } else {
    for (size_t i = 0; i < n; i++) {
      const PipProblem &P = in.h_prob[i];
      cls[i] = plan_one(P);
      est_cells_total += 3ll * (1 + P.nvar * (2 + P.nparm)) + 32;
    }
  }
  s_words = (s_words + 1) & ~1ll;
  s32_words = (s32_words + 1) & ~1ll;
  /* the int32 class leaves shared memory unused at 16 warps per SM: spend it on capacity slack, so
   * fewer problems have to be re-run in a global-memory class */
  const bool s32_wide = try32 && s32_wide_words <= S32_WIDE_MAX_WORDS && getenv("PIPLIB_B200_NO_WIDE_SLACK") == nullptr;
  if (s32_wide) s32_words = (s32_wide_words + 1) & ~1ll;
  /* host descriptors for the rare paths that look at single problems (the whole-grid class) */
  std::vector<PipProblem> fetched_prob;
  auto host_prob = [&]() -> const PipProblem * {
    if (in.h_prob) return in.h_prob;
    if (fetched_prob.empty()) {
      fetched_prob.resize(n);
      CK(cudaMemcpyAsync(fetched_prob.data(), d_prob, n * sizeof(PipProblem), cudaMemcpyDeviceToHost, s));
      CK(cudaStreamSynchronize(s));
    }
    return fetched_prob.data();
  };

  CK(cudaEventRecord(E.ev0, s));
  std::vector<int> order;
  order.reserve(n);
  int round = 0;
  int image_vb = 0, image_elem = -1;     /* arena images built for this value width / pool */
  size_t open_total = n;                /* problems not final yet, all classes */
  for (int k = -2; k < N_G && open_total; k++) {
    int last_open = -1;                 /* problems of this class still open after the previous attempt */
    /* with the reports, problems left open by an attempt with subtree donation (a cell-limit verdict met inside a
     * donated subtree, pip_gather_words_kernel) are solved again without it: that attempt may retire none */
    bool plain = false, redo = false;
    for (int attempt = 0;; attempt++) {
      order.clear();
      for (size_t i = 0; i < n; i++) if (cls[i] == k) order.push_back((int)i);
      if (order.empty()) break;
      const int m = (int)order.size();
      /* every attempt must retire at least one problem (a warp always has room for one worst-case
       * solution): anything else is a scheduling bug, never a verdict */
      if (last_open >= 0 && m >= last_open && !redo)
        throw std::runtime_error("piplib-b200: size class made no progress (" + std::to_string(m) + " problems open)");
      last_open = m;
      const bool identity = (size_t)m == n;           /* every problem of the batch: no permutation needed */
      /* geometry of this round */
      ClassSpec cs;
      int ctas;
      bool team_smem = false;
      if (k < 0) {
        cs.level = (k == -2 && s32_wide) ? PIP_LEVEL_S_WIDE : 2; cs.shared = (k == -2) ? 2 : 1;
        cs.words = std::max<long long>(k == -2 ? s32_words : s_words, 64);
        cs.warps_per_cta = 4;
        cs.stack_words = 1ll << 14;
        size_t smem = (size_t)cs.warps_per_cta * cs.words * sizeof(pip_i64);
        if (smem > E.smem_optin) { cs.warps_per_cta = 1; smem = (size_t)cs.words * sizeof(pip_i64); }
        int per_sm = 1;
        CK(pip_solve_occupancy(cs.shared, cs.warps_per_cta, smem, &per_sm));
        if (per_sm < 1) per_sm = 1;
        ctas = E.sm_count * per_sm;
        int need = (m + cs.warps_per_cta - 1) / cs.warps_per_cta;
        if (ctas > need) ctas = need;
        cs.warps = ctas * cs.warps_per_cta;
      } else {
        cs = G_LADDER[k];
        if (getenv("PIPLIB_B200_NO_TEAM")) cs.team = 0;
        int need_warps = std::min(cs.warps, m);
        /* class M in shared memory: when the working set of every problem of the round at this class's
         * slack fits the SM (e.g. vivien32-shaped cut chains: 22 + 256 rows x 23 words = 56 KB), the CTA's
         * arena is dynamic shared memory instead of global memory */
        if (cs.team && getenv("PIPLIB_B200_NO_TEAM_SMEM") == nullptr) {
          const PipProblem *hp = host_prob();
          long long need = 0;
          for (int q = 0; q < m; q++) {
            const PipProblem &P = hp[order[q]];
            need = std::max(need, pip_layout_words(P.nvar, P.nparm, P.ni, P.nc, P.flags, cs.level, 8));
          }
          need = (need + 1) & ~1ll;
          const size_t bytes = (size_t)need * sizeof(pip_i64);
          if (bytes + 2048 <= E.smem_optin) {
            int per_sm = 0;
            CK(pip_solve_occupancy(4, cs.team, bytes, &per_sm));
            if (per_sm >= 1) {
              team_smem = true;
              cs.words = need;
              need_warps = std::min(m, E.sm_count * per_sm);
            }
          }
        }
        if (cs.team) { ctas = need_warps; cs.warps = ctas; cs.warps_per_cta = cs.team; }
        else {
          ctas = (need_warps + cs.warps_per_cta - 1) / cs.warps_per_cta;
          cs.warps = ctas * cs.warps_per_cta;
        }
      }
      /* cell pool: every warp must be able to hold one worst-case solution */
      long long est = est_cells_total * (long long)m / (long long)n;
      long long per_warp = (est + est / 4) / cs.warps + 1 + in.sol_size;
      if (attempt > 0) per_warp = std::max<long long>(per_warp, 4ll * in.sol_size);
      /* (+ the windows of the hand-over launch, below) */
      const long long per_warp2 = k < 0 ? 3ll * in.sol_size : 0;
      E.d_cells.reserve((size_t)(per_warp + per_warp2) * cs.warps * sizeof(PipCell));
      E.d_stack.reserve((size_t)cs.stack_words * cs.warps * sizeof(pip_i64));
      if (!cs.shared && !team_smem) E.d_gwork.reserve((size_t)cs.words * cs.warps * sizeof(pip_i64));
      if (!identity) {
        E.d_order.reserve((size_t)m * sizeof(int));
        CK(cudaMemcpyAsync(E.d_order.p, order.data(), (size_t)m * sizeof(int), cudaMemcpyHostToDevice, s));
      }
      const int *d_order = identity ? nullptr : (const int *)E.d_order.p;
      if (!stream_out) E.d_off.reserve((size_t)m * sizeof(long long));
      CK(cudaMemsetAsync(E.d_queue.p, 0, 16, s));

      PipLaunch L;
      memset(&L, 0, sizeof L);
      L.prob = d_prob; L.pool = d_pool; L.pool_elem_log2 = elem_log2; L.order = d_order; L.nprob = m;
      L.res = (PipResult *)E.d_res.p;
      L.cells = (PipCell *)E.d_cells.p; L.cells_per_warp = per_warp;
      L.stack = (pip_i64 *)E.d_stack.p; L.stack_words_per_warp = cs.stack_words;
      L.gwork = (cs.shared || team_smem) ? nullptr : (pip_i64 *)E.d_gwork.p;
      L.work_words = (int)cs.words;
      L.queue = (unsigned *)E.d_queue.p;
      L.sol_size = in.sol_size; L.maxcol = in.maxcol; L.maxparm = PIP_MAXPARM;
      L.slack_level = cs.level;
      L.prof = (unsigned long long *)E.d_prof.p;
      /* one shape for the whole batch: carve the arena here, once, instead of once per problem on the device */
      if (in.uniform && getenv("PIPLIB_B200_DEVICE_LAYOUT") == nullptr)
        L.have_layout = pip_layout_compute(in.uniform->nvar, in.uniform->nparm, in.uniform->ni, in.uniform->nc,
                                           in.uniform->flags, cs.level, (int)cs.words, cs.shared == 2 ? 4 : 8, &L.layout);
      /* ... and run the problem load ahead of the solver: arena images, two block copies per problem in the kernel */
      if (L.have_layout && k < 0 && getenv("PIPLIB_B200_NO_IMAGE") == nullptr) {
        const int vb = cs.shared == 2 ? 4 : 8;
        const long long w1 = (L.layout.m.data - L.layout.m.den) + ((long long)in.uniform->ni * L.layout.m.stride * vb + 7) / 8;
        const long long w2 = ((long long)in.uniform->nc * L.layout.cstride * vb + 7) / 8;
        if (image_vb != vb || image_elem != elem_log2) {
          E.d_image.reserve((size_t)n * (size_t)(w1 + w2) * sizeof(pip_i64) + 64);
          CK(pip_launch_image(d_prob, d_pool, elem_log2, (long long)n, &L.layout, (pip_i64 *)E.d_image.p, (int)(w1 + w2), (int)w1, vb, s));
          out.times.launches++;
          image_vb = vb; image_elem = elem_log2;
        }
        L.images = (const pip_i64 *)E.d_image.p; L.image_words = (int)(w1 + w2); L.image_w1 = (int)w1;
      }
      double tk = now_s();
      /* PIPLIB_B200_LARGE_FROM=<class index> moves the hand-over (tests), a negative value disables it */
      const char *lf = getenv("PIPLIB_B200_LARGE_FROM");
      const int large_from = lf && *lf ? atoi(lf) : PIP_LARGE_FROM_DEFAULT;
      bool use_large = large_from >= 0 && k >= large_from && m <= 4 && elem_log2 <= 3;
      if (use_large) { const PipProblem *hp = host_prob(); for (int q = 0; q < m && use_large; q++) use_large = large_eligible(hp[order[q]]); }
      /* word mode: every stream can be written by the solver itself (no column surgery anywhere in the batch):
       * no cells, no decode kernel -- a copy into the compact buffer is all that follows the solve */
      const bool words_round = stream_out && all_sized && !use_large && getenv("PIPLIB_B200_CELL_DECODE") == nullptr;
      L.emit_words = words_round ? 1 : 0;
      /* subtree donation (PipSteal): worth it when the batch is small against the machine -- then the tail of
       * the launch is a few heavy parametric trees and most warps are idle; a big batch balances by problems.
       * PIPLIB_B200_STEAL=0/1 overrides */
      const int dmode = g_donation.load();
      bool steal = words_round && k < 0 &&
                   (dmode > 0 || (dmode < 0 && (long long)m <= 2ll * cs.warps && (!in.uniform || in.uniform->nparm > 0)));
      if (const char *sv = getenv("PIPLIB_B200_STEAL")) steal = words_round && k < 0 && atoi(sv) != 0;
      steal = steal && !plain;
      auto arm_donation = [&](PipSteal &S) {
        S.mode = 1; S.cap = 1 << 16;
        if (const char *cv = getenv("PIPLIB_B200_STEAL_CAP")) S.cap = std::max(1024, atoi(cv));
        E.d_stl_offers.reserve((size_t)S.cap * sizeof(PipOffer));
        E.d_stl_segs.reserve((size_t)S.cap * sizeof(PipResult));
        E.d_stl_next.reserve((size_t)S.cap * sizeof(int));
        E.d_stl_hwm.reserve((size_t)S.cap * sizeof(int));
        E.d_stl_head_next.reserve(n * sizeof(int));
        E.d_stl_head_hwm.reserve(n * sizeof(int));
        E.d_stl_ctl.reserve(PIP_STL_NCTL * sizeof(unsigned));
        CK(cudaMemsetAsync(E.d_stl_offers.p, 0, (size_t)S.cap * sizeof(PipOffer), s));
        CK(cudaMemsetAsync(E.d_stl_head_next.p, 0xff, n * sizeof(int), s));
        CK(cudaMemsetAsync(E.d_stl_head_hwm.p, 0, n * sizeof(int), s));
        CK(cudaMemsetAsync(E.d_stl_ctl.p, 0, PIP_STL_NCTL * sizeof(unsigned), s));
        S.offers = (PipOffer *)E.d_stl_offers.p; S.ctl = (unsigned *)E.d_stl_ctl.p;
        S.segs = (PipResult *)E.d_stl_segs.p; S.seg_next = (int *)E.d_stl_next.p; S.seg_hwm = (int *)E.d_stl_hwm.p;
        S.head_next = (int *)E.d_stl_head_next.p; S.head_hwm = (int *)E.d_stl_head_hwm.p;
      };
      if (steal) arm_donation(L.steal);
      /* heavy-problem hand-over (PipLaunch::budget): a batch balances by problems until its tail, which is a
       * handful of very large trees on one warp each while the machine idles (loop nests: 16 ms of a 41 ms launch
       * at 200 000 problems).  Those stop at `budget` pivots and a second launch, with donation, solves them with
       * many warps.  Not for a batch so big that the tail is noise, nor when other lanes fill the machine anyway.
       * PIPLIB_B200_HEAVY_PIVOTS=<n> sets the budget and forces the hand-over, 0 disables it */
      unsigned heavy_budget = 1536;
      bool handover = words_round && k < 0 && !steal && !in.overlapped && m <= (1 << 19) && (!in.uniform || in.uniform->nparm > 0);
      if (const char *hv = getenv("PIPLIB_B200_HEAVY_PIVOTS")) {
        heavy_budget = (unsigned)atoi(hv);
        handover = words_round && k < 0 && !steal && heavy_budget > 0;
      }
      handover = handover && !plain;
      redo = false;
      PipLaunch L2;
      const PipSteal *gather_stl = steal ? &L.steal : nullptr;
      if (handover) {
        E.d_heavy.reserve((size_t)m * sizeof(int));
        L.budget = heavy_budget;
        L.heavy_max = (unsigned)std::max(64, m / 64);
        L.heavy = (int *)E.d_heavy.p;
        L2 = L;
        L2.budget = 0; L2.from_heavy = 1;
        L2.heavy_warps = 8;
        if (const char *hw = getenv("PIPLIB_B200_HEAVY_WARPS")) L2.heavy_warps = std::max(1, atoi(hw));
        L2.cell_base = per_warp * (long long)cs.warps; L2.cells_per_warp = per_warp2;
        L2.heavy_region = per_warp2 * (long long)cs.warps;
        arm_donation(L2.steal);
        gather_stl = &L2.steal;
      }
      if (use_large) {
        run_large_round(in, host_prob(), d_pool, elem_log2, order, (PipCell *)E.d_cells.p, per_warp, (PipResult *)E.d_res.p, s);
        out.times.launches += m;
      } else {
        CK(pip_launch_solve(&L, (k >= 0 && cs.team) ? (team_smem ? 4 : 3) : cs.shared, ctas, cs.warps_per_cta, s));
        out.times.launches++;
        if (handover) {
          CK(pip_launch_solve(&L2, cs.shared, ctas, cs.warps_per_cta, s));
          out.times.launches++;
        }
      }
      /* this round's output: packed cells, or (device-decode mode) serialised quasts */
      if (ser_mode && (!all_sized || use_large)) {      /* sizing pass, unless the solver sized every stream itself */
        CK(pip_launch_serialize((PipResult *)E.d_res.p, d_order, (const PipCell *)E.d_cells.p, d_parm, in.uniform_decode,
                                nullptr, nullptr, nullptr, m, 0, nullptr, s));
        out.times.launches++;
      }
      long long total = 0;
      int finals = -1;                   /* stream_out: problems of this round with a final status */
      if (stream_out) {
        /* decode with span reservation: no scan, no host round trip before the decode; if the compact
         * buffer turns out too small, grow it and decode the round again (the cells are still there) */
        for (;;) {
          CK(cudaMemsetAsync(so.ctl + PIP_SO_FINALS, 0, 2 * sizeof(unsigned long long), s));   /* finals, overflow */
          if (words_round)
            CK(pip_launch_gather_words((PipResult *)E.d_res.p, d_order, (const PipCell *)E.d_cells.p,
                                       (pip_i64 *)E.d_compact.p, m, &so, gather_stl, in.sol_size, s));
          else
            CK(pip_launch_serialize((PipResult *)E.d_res.p, d_order, (const PipCell *)E.d_cells.p, d_parm, in.uniform_decode,
                                    nullptr, (pip_i64 *)E.d_compact.p, nullptr, m, 1, &so, s));
          out.times.launches++;
          CK(cudaEventRecord(E.ev1, s));
          CK(cudaMemcpyAsync(h_ctl, so.ctl, (PIP_SO_NCTL + PIP_SO_NSTAT) * sizeof(unsigned long long), cudaMemcpyDeviceToHost, s));
          CK(cudaStreamSynchronize(s));
          if (!h_ctl[PIP_SO_OVERFLOW]) break;
          /* h_ctl[SLOTS] = what the rounds so far need in total.  Grow, keep the spans of the earlier rounds,
           * rewind the control block (slot cursor, counters) to the end of the previous round, decode again */
          const long long need = (long long)h_ctl[PIP_SO_SLOTS];
          DevBuf bigger;
          bigger.reserve((size_t)(need + need / 4 + 1024) * sizeof(pip_u64));
          if (slots_done) CK(cudaMemcpyAsync(bigger.p, E.d_compact.p, (size_t)slots_done * sizeof(pip_u64), cudaMemcpyDeviceToDevice, s));
          h_ctl[PIP_SO_SLOTS] = (unsigned long long)slots_done;
          h_ctl[PIP_SO_FINALS] = h_ctl[PIP_SO_OVERFLOW] = h_ctl[3] = 0;
          for (int c = 0; c < PIP_SO_NSTAT; c++) h_ctl[PIP_SO_NCTL + c] = stats_prev[c];
          CK(cudaMemcpyAsync(so.ctl, h_ctl, (PIP_SO_NCTL + PIP_SO_NSTAT) * sizeof(unsigned long long), cudaMemcpyHostToDevice, s));
          CK(cudaStreamSynchronize(s));
          E.d_compact.release();
          E.d_compact = bigger;
          so.cap = (long long)(E.d_compact.cap / sizeof(pip_u64));
        }
        for (int c = 0; c < PIP_SO_NSTAT; c++) stats_prev[c] = h_ctl[PIP_SO_NCTL + c];
        finals = (int)h_ctl[PIP_SO_FINALS];
        total = (long long)h_ctl[PIP_SO_SLOTS] - slots_done;
      } else {
        CK(pip_launch_gather((PipResult *)E.d_res.p, d_order, (const PipCell *)E.d_cells.p,
                             (long long *)E.d_off.p, nullptr, m, (long long *)E.d_total.p, ser_mode ? 2 : 0, s));
        out.times.launches++;
        CK(cudaMemcpyAsync(E.h_total.p, E.d_total.p, sizeof(long long), cudaMemcpyDeviceToHost, s));
        CK(cudaStreamSynchronize(s));
        total = *(long long *)E.h_total.p;
        E.d_compact.reserve((size_t)std::max<long long>(total, 1) * sizeof(pip_u64));
        if (ser_mode)
          CK(pip_launch_serialize((PipResult *)E.d_res.p, d_order, (const PipCell *)E.d_cells.p, d_parm, in.uniform_decode,
                                  (const long long *)E.d_off.p, (pip_i64 *)E.d_compact.p, (pip_u64 *)E.d_hash.p, m, 1,
                                  nullptr, s));
        else
          CK(pip_launch_gather((PipResult *)E.d_res.p, d_order, (const PipCell *)E.d_cells.p,
                               (long long *)E.d_off.p, (pip_u64 *)E.d_compact.p, m, (long long *)E.d_total.p, 1, s));
        out.times.launches++;
        CK(cudaEventRecord(E.ev1, s));
        CK(cudaStreamSynchronize(s));
      }
      out.times.kernel += now_s() - tk;
      if (round < 8) { out.times.round_s[round] = (float)(now_s() - tk); out.times.round_n[round] = m; }
      const double t_round = now_s() - tk;
      int pending = 0, escalated = 0;
      if (stream_out && finals == m) {
        /* the common case: every problem of the round is final -- nothing per problem crosses PCIe */
        for (int q = 0; q < m; q++) cls[order[q]] = 1000;
        slots_done += total;
        open_total -= (size_t)m;
        round++;
        out.times.rounds++;
      } else {
        /* fetch records (+ cells) */
        double td = now_s();
        need_h_res();
        CK(cudaMemcpyAsync(h_res, E.d_res.p, n * sizeof(PipResult), cudaMemcpyDeviceToHost, s));
        out.times.d2h_bytes += n * sizeof(PipResult);
        PinBuf *chunk = nullptr;
        if (!stream_out) {
          if ((size_t)round >= E.h_chunks.size()) E.h_chunks.resize(round + 1);
          chunk = &E.h_chunks[round];
          if (in.fetch_cells && total > 0) {
            chunk->reserve((size_t)total * sizeof(pip_u64));
            CK(cudaMemcpyAsync(chunk->p, E.d_compact.p, (size_t)total * sizeof(pip_u64), cudaMemcpyDeviceToHost, s));
            out.times.d2h_bytes += (size_t)total * sizeof(pip_u64);
          }
        }
        CK(cudaStreamSynchronize(s));
        out.times.d2h += now_s() - td;
        slots_done += total;
        round++;
        out.times.rounds++;
        /* classify */
        bool widened_input = false;
        for (int q = 0; q < m; q++) {
          const int i = order[q];
          const PipResult &r = h_res[i];
          if (r.status == PIP_ST_PENDING) { pending++; continue; }
          if (r.status == PIP_ST_WIDEN) { cls[i] = -1; h_res[i].status = PIP_ST_PENDING; escalated++; widened_input = true; continue; }
          if (r.status == PIP_ST_CAPACITY && k + 1 < N_G && !use_large) {   /* class L has no larger class above it */
            /* the wide int32 class already has half of G3's cut rows and all of its context rows: what
             * outgrew it goes straight to the first team class (4x the rows) instead of failing G3 too */
            cls[i] = k < 0 ? ((k == -2 && s32_wide) ? 1 : 0) : k + 1;
            h_res[i].status = PIP_ST_PENDING;
            escalated++;
            continue;
          }
          cls[i] = 1000;                       /* final */
          open_total--;
          if (!stream_out) {
            out.res[i] = r;
            out.base[i] = (const pip_u64 *)chunk->p;
          }
        }
        /* a problem whose input did not fit the int32 pool: from now on every round reads the int64 pool */
        if (widened_input && elem_log2 < 3 && in.widen_pool) {
          d_pool = in.widen_pool(in.widen_ctx, s);
          elem_log2 = 3;
        }
        if (pending || escalated) {
          /* re-arm the open problems on the device */
          CK(cudaMemcpyAsync(E.d_res.p, h_res, n * sizeof(PipResult), cudaMemcpyHostToDevice, s));
          CK(cudaStreamSynchronize(s));
        }
      }
      if (getenv("PIPLIB_B200_TIMING"))
        fprintf(stderr, "[piplib-b200] round %d: class %d attempt %d, %d problems on %d warps (%d words/warp): %.3f s, %d not final (%d pending)%s%s\n",
                round - 1, k, attempt, m, cs.warps, (int)cs.words, t_round, escalated + pending, pending, use_large ? " [whole-grid kernel]" : "",
                team_smem ? " [team arena in shared memory]" : "");
      if (pending == 0) break;
      if (in.want_info && stream_out && (steal || handover) && !plain) plain = redo = true;
    }
  }
  CK(cudaEventElapsedTime(&out.times.device_ms, E.ev0, E.ev1));
  if (stream_out) {
    out.dev.words = (const pip_i64 *)E.d_compact.p;
    out.dev.slots = slots_done;
    out.dev.status = so.status; out.dev.hash = so.hash; out.dev.off = so.off; out.dev.len = so.len; out.dev.info = so.info;
    for (int k = 0; k < PIP_SO_NSTAT; k++) out.dev.stats[k] = h_ctl[PIP_SO_NCTL + k];
    /* anything still unsolved is too large for the ladder: its status array entry says CAPACITY already
     * (the last decode pass wrote the record's status) */
  } else {
    if (ser_mode) {
      E.h_hash.reserve(n * sizeof(pip_u64));
      CK(cudaMemcpy(E.h_hash.p, E.d_hash.p, n * sizeof(pip_u64), cudaMemcpyDeviceToHost));
      out.hashes.assign((const pip_u64 *)E.h_hash.p, (const pip_u64 *)E.h_hash.p + n);
      out.times.d2h_bytes += n * sizeof(pip_u64);
    }
    /* anything still unsolved is too large for the ladder */
    for (size_t i = 0; i < n; i++)
      if (cls[i] != 1000) { out.res[i] = PipResult(); out.res[i].status = PIP_ST_CAPACITY; }
  }
#ifdef PIP_PROFILE
  CK(cudaMemcpy(out.times.phase_cycles, E.d_prof.p, sizeof(unsigned long long) * PIP_NPHASE, cudaMemcpyDeviceToHost));
#endif
  out.times.total = now_s() - t_begin;
}
