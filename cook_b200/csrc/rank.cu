// rank.cu — DRU fair-share ranking on the GPU (SURVEY §8a R1-R7).
//
// Replaces sort-jobs-by-dru-helper (scheduler/scheduler.clj:2073-2091),
// limit-over-quota-jobs (:2057-2071), dru/compute-task-scored-task-pairs
// (dru.clj:50-80), dru/sorted-merge (dru.clj:82-104), filter-based-on-quota
// (scheduler.clj:2134-2157) and filter-offensive-jobs (:2198-2229).
//
// Pipeline (all on the pool's stream, no host round trips):
//   K1 iota + comparator sort by (user name rank, -priority, start, task id,
//      job id)                      -> per-user segments in tools.clj:614-641 order
//   K2 segment bounds
//   K3 warp-per-user fold           -> cumulative usage in the reference's
//      left-fold order (lane-serial shuffle chain keeps f64 association),
//      over-quota truncation, DRU = max(mem/div, cpus/div) (IEEE div.rn.f64)
//   K4 comparator sort of positions by (dru, k-way-merge tie rule)
//   K5 single-warp queue filter     -> pending only, pool quota, group quota,
//      offensive filter, stable compaction.
#include "common.cuh"
#include "sort.cuh"

namespace {

struct TaskCols {
  const int32_t* user;
  const int32_t* prio;
  const int64_t* start;
  const int64_t* tid;
  const int64_t* jid;
  const double* cpus;
  const double* mem;
  const double* gpus;
};

// tools.clj:614-641 compare of feature vectors, prefixed by the user's name
// rank so that one global sort yields all per-user lists, users in name order.
struct LessUserTask {
  TaskCols t;
  const int32_t* name_rank;
  __device__ bool operator()(int32_t a, int32_t b) const {
    int ua = name_rank[t.user[a]], ub = name_rank[t.user[b]];
    if (ua != ub) return ua < ub;
    int pa = -t.prio[a], pb = -t.prio[b];
    if (pa != pb) return pa < pb;
    long long sa = t.start[a], sb = t.start[b];
    if (sa != sb) return sa < sb;
    long long ta = t.tid[a], tb = t.tid[b];
    if (ta != tb) return ta < tb;
    long long ja = t.jid[a], jb = t.jid[b];
    if (ja != jb) return ja < jb;
    return a < b;
  }
};

// Global emission order of dru/sorted-merge (dru.clj:82-104).  X, Y are
// positions in the user-sorted array.  The merge emits, at every step, the head
// with the smallest (dru, -arrival, name) where arrival = step at which the
// user's previous task was emitted (0 for a user's first task): the popped
// user's remainder is consed to the FRONT before a STABLE re-sort (:93-94).
// A popped user whose next task has the same dru is therefore popped again: a
// user's RUN of equal-dru tasks (run_start) is emitted as one block, and the
// blocks of one dru value go in the order their heads held when the first of
// them came up.  Hence for equal dru:  X before Y  <=>  the task before X's run
// was emitted AFTER the task before Y's run, which recurses on those two tasks
// (smaller dru) with the roles swapped.  (Comparing prev(X) with prev(Y) instead
// is only right for runs of one task: with a longer run, X's whole run goes out
// before a later-arriving Y even becomes a head.)
struct LessMerge {
  const double* dru;        // by sorted position; NaN = cut by limit-over-quota
  const int32_t* user_at;   // user of sorted position
  const int32_t* seg_start; // per user
  const int32_t* name_rank;
  const int32_t* run_start; // by sorted position: first position of its user's run of equal dru
  __device__ bool operator()(int32_t x, int32_t y) const {
    double dx = dru[x], dy = dru[y];
    bool kx = dx == dx, ky = dy == dy;
    if (kx != ky) return kx;  // truncated tasks sort last
    if (!kx) return x < y;
    while (true) {
      if (dx != dy) return dx < dy;
      int ux = user_at[x], uy = user_at[y];
      if (ux == uy) return x < y;  // same user: queue order
      const int rx = run_start[x], ry = run_start[y];
      bool hx = rx > seg_start[ux], hy = ry > seg_start[uy];
      if (!hx && !hy) return name_rank[ux] < name_rank[uy];
      if (!hx) return false;  // X's run has arrival 0 => Y first
      if (!hy) return true;
      // before(X,Y) = before(prev(run(Y)), prev(run(X))): swap roles and step back
      x = ry - 1; y = rx - 1;
      dx = dru[x]; dy = dru[y];
    }
  }
};

// run_start for LessMerge: an inclusive max-scan of "p starts a run" (first slot of the user's segment,
// or a dru different from the slot before; NaN never equals) over the user-sorted positions.  Tiles of
// RS_TB, one short serial pass over the tile maxima, then the fix-up.
constexpr int RS_TB = 1024;
__global__ void __launch_bounds__(RS_TB) run_start_tiles(const double* __restrict__ dru_at, const int32_t* __restrict__ user_at,
                                                          const int32_t* __restrict__ seg_start, int n,
                                                          int32_t* __restrict__ run_start, int32_t* __restrict__ tile_max) {
  __shared__ int wmax[RS_TB / 32];
  const int p = blockIdx.x * RS_TB + threadIdx.x, lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  int v = 0;
  if (p < n) v = (p == seg_start[user_at[p]] || !(dru_at[p - 1] == dru_at[p])) ? p : 0;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) { const int y = __shfl_up_sync(0xffffffffu, v, o); if (lane >= o) v = max(v, y); }
  if (lane == 31) wmax[w] = v;
  __syncthreads();
  if (w == 0) {
    int t = wmax[lane];
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const int y = __shfl_up_sync(0xffffffffu, t, o); if (lane >= o) t = max(t, y); }
    wmax[lane] = t;
  }
  __syncthreads();
  if (w) v = max(v, wmax[w - 1]);
  if (p < n) run_start[p] = v;
  if (threadIdx.x == RS_TB - 1) tile_max[blockIdx.x] = v;
}
__global__ void run_start_carry(int32_t* tile_max, int nb) {   // one thread: exclusive prefix max
  int m = 0;
  for (int b = 0; b < nb; b++) { const int t = tile_max[b]; tile_max[b] = m; m = max(m, t); }
}
__global__ void __launch_bounds__(RS_TB) run_start_fix(int32_t* run_start, const int32_t* tile_max, int n) {
  const int p = blockIdx.x * RS_TB + threadIdx.x;
  if (p < n) run_start[p] = max(run_start[p], tile_max[blockIdx.x]);
}

__global__ void scatter_dru_kernel(const int32_t* __restrict__ idx, const double* __restrict__ dru_at,
                                   int n, double* __restrict__ dru_task) {
  int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p < n) dru_task[idx[p]] = dru_at[p];
}

__global__ void iota_kernel(int32_t* p, int n) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = i;
}

__global__ void seg_bounds_kernel(const int32_t* __restrict__ idx, const int32_t* __restrict__ user,
                                  int n, int32_t* seg_start, int32_t* seg_end,
                                  int32_t* user_at) {
  int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= n) return;
  int u = user[idx[p]];
  user_at[p] = u;
  if (p == 0 || user[idx[p - 1]] != u) seg_start[u] = p;
  if (p == n - 1 || user[idx[p + 1]] != u) seg_end[u] = p + 1;
}

struct UserCols {
  const double *div_mem, *div_cpus, *div_gpus;
  const double *q_count, *q_cpus, *q_mem, *q_gpus;
};

// K3: one warp per user.  Lane-serial fold keeps the reference's left-fold
// association: acc = ((acc + x0) + x1) + ... exactly as `reductions` does.
__global__ void __launch_bounds__(128) user_fold_kernel(
    const int32_t* __restrict__ idx, TaskCols t, UserCols uc, const int32_t* __restrict__ seg_start,
    const int32_t* __restrict__ seg_end, int n_users, int dru_mode, int max_over_quota,
    double* __restrict__ dru_at, int32_t* n_kept_total, const GridFlag* gf, int n_scan) {
  if (n_scan > 0 && grid_exact(gf, n_scan)) return;   // the order-wide scans below did it
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (warp >= n_users) return;
  const int u = warp;
  const int s = seg_start[u], e = seg_end[u];
  if (e <= s) return;
  const double md = uc.div_mem[u], cd = uc.div_cpus[u], gd = uc.div_gpus[u];
  const double qn = uc.q_count[u], qc = uc.q_cpus[u], qm = uc.q_mem[u], qg = uc.q_gpus[u];
  // The three cumulative sums are independent serial chains: lanes 0..2 run one each over
  // the batch staged in shared memory (carried in `acc`), then every lane reads its prefix.
  __shared__ double fold_s[4][3][32];
  double (*fs)[32] = fold_s[threadIdx.x >> 5];
  double acc = 0.0;
  double am = 0.0, ac = 0.0, ag = 0.0;   // carries of the scan path
  const bool exact = grid_exact(gf, e - s);   // every partial sum is exact: a parallel scan gives the left fold's bits
  int over = 0;
  bool cut = false;
  int kept = 0;
  const double NaN = __longlong_as_double(0x7ff8000000000000LL);
  auto chunk = [&](const int base, const double xm, const double xc, const double xg) {
    const int p = base + lane;
    double mym, myc, myg;
    if (exact) {
      mym = am + warp_incl_scan(xm, lane); myc = ac + warp_incl_scan(xc, lane); myg = ag + warp_incl_scan(xg, lane);
      am = __shfl_sync(0xffffffffu, mym, 31); ac = __shfl_sync(0xffffffffu, myc, 31); ag = __shfl_sync(0xffffffffu, myg, 31);
    } else {
      fs[0][lane] = xm; fs[1][lane] = xc; fs[2][lane] = xg;
      __syncwarp();
      int cntn = min(32, e - base);
      if (lane < 3) {
        double* row = fs[lane];
#pragma unroll 8
        for (int l = 0; l < cntn; l++) { acc = acc + row[l]; row[l] = acc; }
      }
      __syncwarp();
      mym = fs[0][lane]; myc = fs[1][lane]; myg = fs[2][lane];
      __syncwarp();
    }
    // scheduler.clj:2057-2071: keep while #violating prefixes <= limit
    bool viol = false;
    if (p < e) {
      double cnt = (double)(p - s + 1);
      viol = !(cnt <= qn && myc <= qc && mym <= qm && myg <= qg);
    }
    unsigned vb = __ballot_sync(0xffffffffu, viol);
    int over_incl = over + __popc(vb & (0xffffffffu >> (31 - lane)));
    bool keep = (p < e) && !cut && (over_incl <= max_over_quota);
    double d = NaN;
    if (keep) {
      if (dru_mode == 0) {
        double a = mym / md, b = myc / cd;
        d = a > b ? a : b;
      } else {
        d = myg / gd;
      }
    }
    if (p < e) dru_at[p] = d;
    unsigned kb = __ballot_sync(0xffffffffu, keep);
    kept += __popc(kb);
    over += __popc(vb);
    if (over > max_over_quota) cut = true;  // later batches are all beyond the cut
  };
  if (exact) {
    // the gathers (idx -> amounts) are what a long segment waits for: four chunks in flight
    for (int base = s; base < e; base += 128) {
      double xm4[4], xc4[4], xg4[4];
#pragma unroll
      for (int q = 0; q < 4; q++) {
        const int p = base + 32 * q + lane;
        xm4[q] = xc4[q] = xg4[q] = 0.0;
        if (p < e) { const int ti = idx[p]; xm4[q] = t.mem[ti]; xc4[q] = t.cpus[ti]; xg4[q] = t.gpus[ti]; }
      }
#pragma unroll
      for (int q = 0; q < 4; q++)
        if (base + 32 * q < e) chunk(base + 32 * q, xm4[q], xc4[q], xg4[q]);
    }
  } else {
    for (int base = s; base < e; base += 32) {
      const int p = base + lane;
      double xm = 0.0, xc = 0.0, xg = 0.0;
      if (p < e) { const int ti = idx[p]; xm = t.mem[ti]; xc = t.cpus[ti]; xg = t.gpus[ti]; }
      chunk(base, xm, xc, xg);
    }
  }
  if (lane == 0 && kept) atomicAdd(n_kept_total, kept);
}

// K3 for exact-grid amounts (common.cuh: any association gives the left fold's bits): the per-user
// running sums are ONE inclusive scan over the whole sorted order minus the scan just before the
// user's first slot, the over-quota count is a second scan over the violation flags.  No user, however
// long its list, sits on one warp.  Five launches: amount tiles, their totals, violation tiles, their
// totals, the finish (keep / dru / kept count).
constexpr int OS_TB = 256, OS_IPT = 8, OS_TILE = OS_TB * OS_IPT;

struct OrderScan {
  const int32_t* idx; TaskCols t; UserCols uc;
  const int32_t* user_at; const int32_t* seg_start;
  int n, dru_mode, max_over_quota;
  const GridFlag* gf;
  double *pm, *pc, *pg;      // [n] tile-local inclusive sums
  double *bm, *bc, *bg;      // [tiles] totals, then exclusive offsets
  int32_t* pv; int32_t* bv;  // the same for the violation flags
  double* dru_at; int32_t* n_kept_total;
};

__device__ __forceinline__ void os_user_sums(const OrderScan& a, int p, int s, double& m, double& c, double& g) {
  const int tp = p / OS_TILE;
  m = a.pm[p] + a.bm[tp]; c = a.pc[p] + a.bc[tp]; g = a.pg[p] + a.bg[tp];
  if (s > 0) {
    const int ts = (s - 1) / OS_TILE;
    m = m - (a.pm[s - 1] + a.bm[ts]); c = c - (a.pc[s - 1] + a.bc[ts]); g = g - (a.pg[s - 1] + a.bg[ts]);
  }
}

__global__ void __launch_bounds__(OS_TB) os_amount_tiles(OrderScan a) {
  if (!grid_exact(a.gf, a.n)) return;
  __shared__ double s_m[OS_TB / 32], s_c[OS_TB / 32], s_g[OS_TB / 32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int p0 = blockIdx.x * OS_TILE + threadIdx.x * OS_IPT;
  double xm[OS_IPT], xc[OS_IPT], xg[OS_IPT];
#pragma unroll
  for (int k = 0; k < OS_IPT; k++) {
    const int p = p0 + k;
    xm[k] = xc[k] = xg[k] = 0.0;
    if (p < a.n) { const int ti = a.idx[p]; xm[k] = a.t.mem[ti]; xc[k] = a.t.cpus[ti]; xg[k] = a.t.gpus[ti]; }
  }
#pragma unroll
  for (int k = 1; k < OS_IPT; k++) { xm[k] = xm[k - 1] + xm[k]; xc[k] = xc[k - 1] + xc[k]; xg[k] = xg[k - 1] + xg[k]; }
  const double im = warp_incl_scan(xm[OS_IPT - 1], lane), ic = warp_incl_scan(xc[OS_IPT - 1], lane),
               ig = warp_incl_scan(xg[OS_IPT - 1], lane);
  if (lane == 31) { s_m[warp] = im; s_c[warp] = ic; s_g[warp] = ig; }
  __syncthreads();
  double om = im - xm[OS_IPT - 1], oc = ic - xc[OS_IPT - 1], og = ig - xg[OS_IPT - 1];
  for (int w = 0; w < warp; w++) { om = om + s_m[w]; oc = oc + s_c[w]; og = og + s_g[w]; }
#pragma unroll
  for (int k = 0; k < OS_IPT; k++) {
    const int p = p0 + k;
    if (p < a.n) { a.pm[p] = om + xm[k]; a.pc[p] = oc + xc[k]; a.pg[p] = og + xg[k]; }
  }
  if (threadIdx.x == OS_TB - 1) {
    a.bm[blockIdx.x] = om + xm[OS_IPT - 1]; a.bc[blockIdx.x] = oc + xc[OS_IPT - 1]; a.bg[blockIdx.x] = og + xg[OS_IPT - 1];
  }
}

__global__ void os_amount_totals(OrderScan a, int nb) {   // one warp: totals -> exclusive offsets
  if (!grid_exact(a.gf, a.n)) return;
  const int lane = threadIdx.x;
  double am = 0.0, ac = 0.0, ag = 0.0;
  for (int base = 0; base < nb; base += 32) {
    const int b = base + lane;
    const double xm = b < nb ? a.bm[b] : 0.0, xc = b < nb ? a.bc[b] : 0.0, xg = b < nb ? a.bg[b] : 0.0;
    const double im = am + warp_incl_scan(xm, lane), ic = ac + warp_incl_scan(xc, lane), ig = ag + warp_incl_scan(xg, lane);
    if (b < nb) { a.bm[b] = im - xm; a.bc[b] = ic - xc; a.bg[b] = ig - xg; }
    am = __shfl_sync(0xffffffffu, im, 31); ac = __shfl_sync(0xffffffffu, ic, 31); ag = __shfl_sync(0xffffffffu, ig, 31);
  }
}

// scheduler.clj:2057-2071: a prefix violates when (count, cpus, mem, gpus) is not within the quota
__global__ void __launch_bounds__(OS_TB) os_violation_tiles(OrderScan a) {
  if (!grid_exact(a.gf, a.n)) return;
  __shared__ int s_v[OS_TB / 32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int p0 = blockIdx.x * OS_TILE + threadIdx.x * OS_IPT;
  int v[OS_IPT];
#pragma unroll
  for (int k = 0; k < OS_IPT; k++) {
    const int p = p0 + k;
    v[k] = 0;
    if (p < a.n) {
      const int u = a.user_at[p], s = a.seg_start[u];
      double m, c, g;
      os_user_sums(a, p, s, m, c, g);
      const double cnt = (double)(p - s + 1);
      v[k] = !(cnt <= a.uc.q_count[u] && c <= a.uc.q_cpus[u] && m <= a.uc.q_mem[u] && g <= a.uc.q_gpus[u]) ? 1 : 0;
    }
  }
#pragma unroll
  for (int k = 1; k < OS_IPT; k++) v[k] += v[k - 1];
  int iv = v[OS_IPT - 1];
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) { const int y = __shfl_up_sync(0xffffffffu, iv, o); if (lane >= o) iv += y; }
  if (lane == 31) s_v[warp] = iv;
  __syncthreads();
  int ov = iv - v[OS_IPT - 1];
  for (int w = 0; w < warp; w++) ov += s_v[w];
#pragma unroll
  for (int k = 0; k < OS_IPT; k++) {
    const int p = p0 + k;
    if (p < a.n) a.pv[p] = ov + v[k];
  }
  if (threadIdx.x == OS_TB - 1) a.bv[blockIdx.x] = ov + v[OS_IPT - 1];
}

__global__ void os_violation_totals(OrderScan a, int nb) {
  if (!grid_exact(a.gf, a.n)) return;
  const int lane = threadIdx.x;
  int acc = 0;
  for (int base = 0; base < nb; base += 32) {
    const int b = base + lane;
    const int x = b < nb ? a.bv[b] : 0;
    int iv = x;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const int y = __shfl_up_sync(0xffffffffu, iv, o); if (lane >= o) iv += y; }
    iv += acc;
    if (b < nb) a.bv[b] = iv - x;
    acc = __shfl_sync(0xffffffffu, iv, 31);
  }
}

__global__ void __launch_bounds__(OS_TB) os_finish(OrderScan a) {
  if (!grid_exact(a.gf, a.n)) return;
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  bool keep = false;
  if (p < a.n) {
    const int u = a.user_at[p], s = a.seg_start[u];
    int over = a.pv[p] + a.bv[p / OS_TILE];
    if (s > 0) over -= a.pv[s - 1] + a.bv[(s - 1) / OS_TILE];
    keep = over <= a.max_over_quota;
    double d = __longlong_as_double(0x7ff8000000000000LL);
    if (keep) {
      double m, c, g;
      os_user_sums(a, p, s, m, c, g);
      if (a.dru_mode == 0) {
        const double x = m / a.uc.div_mem[u], y = c / a.uc.div_cpus[u];
        d = x > y ? x : y;
      } else {
        d = g / a.uc.div_gpus[u];
      }
    }
    a.dru_at[p] = d;
  }
  const int kept = __syncthreads_count(keep);
  if (threadIdx.x == 0 && kept) atomicAdd(a.n_kept_total, kept);
}

struct QueueFilterArgs {
  const int32_t* pos_sorted;  // positions (into user-sorted array) in merge order
  const int32_t* idx;         // sorted position -> combined task index
  const int32_t* n_kept;      // device: tasks that survived limit-over-quota-jobs
  int R;                      // running count (combined index >= R => pending)
  const double* cpus;         // combined columns
  const double* mem;
  const double* gpus;
  int filter_offensive;
  double off_mem, off_cpus;
  int32_t* out_order;         // combined task index per emitted task
  int32_t* out_ranked;        // pending indices surviving all filters
  int32_t* out_n;
  // queue-order scratch (one entry per emitted task)
  int32_t* ti_at;
  uint8_t* flag;              // pending job still in the queue after the filters so far
  double *xc, *xm, *xg;       // its request (0 for running tasks)
  int32_t* blk_cnt;           // per block of QF_TB entries: survivors, then exclusive offsets
};

constexpr int QF_TB = 256;

// Σ running usage of the pool (scheduler.clj:2118-2123) in input order.
__global__ void pool_usage_kernel(const double* cpus, const double* mem, const double* gpus, int R,
                                  double* out4, const GridFlag* gf) {
  // single warp, lane-serial fold => left-fold association (any association when the sums are exact)
  const int lane = threadIdx.x;
  double ac = 0.0, am = 0.0, ag = 0.0;
  if (grid_exact(gf, R)) {
    for (int i = lane; i < R; i += 32) { ac += cpus[i]; am += mem[i]; ag += gpus[i]; }
    for (int o = 16; o > 0; o >>= 1) {
      ac += __shfl_xor_sync(0xffffffffu, ac, o); am += __shfl_xor_sync(0xffffffffu, am, o); ag += __shfl_xor_sync(0xffffffffu, ag, o);
    }
    if (lane == 0) { out4[0] = (double)R; out4[1] = ac; out4[2] = am; out4[3] = ag; }
    return;
  }
  for (int base = 0; base < R; base += 32) {
    int i = base + lane;
    double xc = i < R ? cpus[i] : 0.0, xm = i < R ? mem[i] : 0.0, xg = i < R ? gpus[i] : 0.0;
    int cntn = min(32, R - base);
    for (int l = 0; l < cntn; l++) {
      ac = ac + __shfl_sync(0xffffffffu, xc, l);
      am = am + __shfl_sync(0xffffffffu, xm, l);
      ag = ag + __shfl_sync(0xffffffffu, xg, l);
    }
  }
  if (lane == 0) { out4[0] = (double)R; out4[1] = ac; out4[2] = am; out4[3] = ag; }
}

// K5 step 1: the merged order as task indices, with each pending job's request
// laid out in queue order so that the sequential filters below stream it.
__global__ void __launch_bounds__(QF_TB) qf_gather_kernel(QueueFilterArgs a) {
  const int i = blockIdx.x * QF_TB + threadIdx.x;
  if (i >= *a.n_kept) return;
  const int ti = a.idx[a.pos_sorted[i]];
  if (a.out_order) a.out_order[i] = ti;
  const bool pend = ti >= a.R;
  a.ti_at[i] = ti;
  a.flag[i] = pend;
  a.xc[i] = pend ? a.cpus[ti] : 0.0;
  a.xm[i] = pend ? a.mem[ti] : 0.0;
  a.xg[i] = pend ? a.gpus[ti] : 0.0;
}

// K5 step 2, once per enabled quota (pool, then quota group): tools.clj:654-668
// filter-sequential -- the usage advances for every job that reaches the filter,
// kept or not, in queue order, with the reference's left-fold association.  The
// four running sums are four independent serial chains: one thread each over a
// chunk staged in shared memory (a job that did not reach the filter adds 0.0,
// which leaves a sum unchanged); everything else is parallel.
constexpr int QF_CH = 1024;
__global__ void __launch_bounds__(QF_CH) qf_quota_kernel(QueueFilterArgs a, cook_pool_quota q,
                                                         const double* usage4, const GridFlag* gf) {
  __shared__ double s[4][QF_CH];
  const int tid = threadIdx.x, n = *a.n_kept;
  const int chain = tid >> 5;                       // chain k runs on lane 0 of warp k
  if (grid_exact(gf, n, fmax(fmax(usage4[0], usage4[1]), fmax(usage4[2], usage4[3]))) &&
      grid_value_ok(usage4[0]) && grid_value_ok(usage4[1]) && grid_value_ok(usage4[2]) && grid_value_ok(usage4[3])) {
    // every partial sum is exact: block-wide parallel scan of the four running sums, carried chunk to chunk
    __shared__ double wsum[4][32];
    const int lane = tid & 31, w = tid >> 5;
    double carry[4] = {usage4[0], usage4[1], usage4[2], usage4[3]};
    for (int base = 0; base < n; base += QF_CH) {
      const int i = base + tid;
      const bool f = i < n && a.flag[i];
      double x[4] = {f ? 1.0 : 0.0, f ? a.xc[i] : 0.0, f ? a.xm[i] : 0.0, f ? a.xg[i] : 0.0};
#pragma unroll
      for (int k = 0; k < 4; k++) { x[k] = warp_incl_scan(x[k], lane); if (lane == 31) wsum[k][w] = x[k]; }
      __syncthreads();
      if (w < 4) { const double t = warp_incl_scan(wsum[w][lane], lane); wsum[w][lane] = t; }
      __syncthreads();
      bool ok = true;
#pragma unroll
      for (int k = 0; k < 4; k++) x[k] = carry[k] + ((w ? wsum[k][w - 1] : 0.0) + x[k]);
      ok = x[0] <= q.count && x[1] <= q.cpus && x[2] <= q.mem && x[3] <= q.gpus;
      if (f && !ok) a.flag[i] = 0;
#pragma unroll
      for (int k = 0; k < 4; k++) carry[k] = carry[k] + wsum[k][31];
      __syncthreads();
    }
    return;
  }
  double acc = (tid & 31) == 0 && chain < 4 ? usage4[chain] : 0.0;
  for (int base = 0; base < n; base += QF_CH) {
    const int i = base + tid, cnt = min(QF_CH, n - base);
    bool f = false;
    if (i < n) {
      f = a.flag[i];
      s[0][tid] = f ? 1.0 : 0.0;
      s[1][tid] = f ? a.xc[i] : 0.0;
      s[2][tid] = f ? a.xm[i] : 0.0;
      s[3][tid] = f ? a.xg[i] : 0.0;
    }
    __syncthreads();
    if ((tid & 31) == 0 && chain < 4) {
      double* row = s[chain];
#pragma unroll 8
      for (int j = 0; j < cnt; j++) { acc = acc + row[j]; row[j] = acc; }
    }
    __syncthreads();
    if (f && !(s[0][tid] <= q.count && s[1][tid] <= q.cpus && s[2][tid] <= q.mem && s[3][tid] <= q.gpus))
      a.flag[i] = 0;
    __syncthreads();
  }
}

// K5 step 3: offensive-job filter (scheduler.clj:2198-2229) and order-preserving
// compaction of the survivors: per-block counts, one scan, scatter.
__global__ void __launch_bounds__(QF_TB) qf_count_kernel(QueueFilterArgs a) {
  const int i = blockIdx.x * QF_TB + threadIdx.x, n = *a.n_kept;
  bool keep = false;
  if (i < n) {
    keep = a.flag[i];
    if (keep && a.filter_offensive && (a.xm[i] > a.off_mem || a.xc[i] > a.off_cpus)) {
      keep = false;
      a.flag[i] = 0;
    }
  }
  const int c = __syncthreads_count(keep);
  if (threadIdx.x == 0) a.blk_cnt[blockIdx.x] = c;
}

__global__ void __launch_bounds__(1024) qf_scan_kernel(QueueFilterArgs a, int nblk_max) {
  __shared__ int wsum[32];
  __shared__ int carry_s;
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  const int nblk = (*a.n_kept + QF_TB - 1) / QF_TB;
  if (tid == 0) carry_s = 0;
  __syncthreads();
  for (int base = 0; base < nblk && base < nblk_max; base += 1024) {
    const int b = base + tid;
    const int v = b < nblk ? a.blk_cnt[b] : 0;
    int x = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { int y = __shfl_up_sync(0xffffffffu, x, o); if (lane >= o) x += y; }
    if (lane == 31) wsum[w] = x;
    __syncthreads();
    if (w == 0) {
      int t = wsum[lane];
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) { int y = __shfl_up_sync(0xffffffffu, t, o); if (lane >= o) t += y; }
      wsum[lane] = t;
    }
    __syncthreads();
    const int carry = carry_s;
    const int incl = x + (w ? wsum[w - 1] : 0);
    if (b < nblk) a.blk_cnt[b] = carry + incl - v;
    __syncthreads();
    if (tid == 1023) carry_s = carry + incl;
    __syncthreads();
  }
  if (tid == 0) *a.out_n = carry_s;
}

__global__ void __launch_bounds__(QF_TB) qf_scatter_kernel(QueueFilterArgs a) {
  __shared__ int wcnt[QF_TB / 32];
  const int i = blockIdx.x * QF_TB + threadIdx.x, n = *a.n_kept;
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const bool keep = i < n && a.flag[i];
  const unsigned kb = __ballot_sync(0xffffffffu, keep);
  if (lane == 0) wcnt[w] = __popc(kb);
  __syncthreads();
  if (blockIdx.x * QF_TB >= n) return;
  int off = a.blk_cnt[blockIdx.x];
  for (int k = 0; k < w; k++) off += wcnt[k];
  if (keep) a.out_ranked[off + __popc(kb & ((1u << lane) - 1u))] = a.ti_at[i] - a.R;
}

template <class T>
cudaError_t upload2(Arena& ar, cudaStream_t st, const T* a, int na, const T* b, int nb, T** out) {
  T* d = ar.take<T>((size_t)na + nb + 1);
  if (!d) return cudaErrorMemoryAllocation;
  *out = d;
  cudaError_t e = cudaSuccess;
  if (na) e = cudaMemcpyAsync(d, a, sizeof(T) * na, cudaMemcpyHostToDevice, st);
  if (e != cudaSuccess) return e;
  if (nb) e = cudaMemcpyAsync(d + na, b, sizeof(T) * nb, cudaMemcpyHostToDevice, st);
  return e;
}

}  // namespace

extern "C" int32_t cook_rank(cook_pool* pool, const cook_tasks_soa* running,
                             const cook_tasks_soa* pending, const cook_user_table* users,
                             const cook_pool_quota* pool_quota, const cook_pool_quota* group_quota,
                             const double* group_usage, const cook_rank_params* params,
                             int32_t* out_ranked_idx, int32_t* out_n, double* out_dru,
                             int32_t* out_order, int32_t* out_order_n) {
  if (!pool) return COOK_E_BADARG;
  if (!running || !pending || !users || !params || !out_ranked_idx || !out_n)
    return set_err(pool, COOK_E_BADARG, "cook_rank: null argument");
  const int R = running->n, J = pending->n, N = R + J, U = users->n_users;
  if (R < 0 || J < 0 || U <= 0) return set_err(pool, COOK_E_BADARG, "cook_rank: bad sizes");
  if (!idx_in_range(running->user, R, 0, U) || !idx_in_range(pending->user, J, 0, U))
    return set_err(pool, COOK_E_BADARG, "cook_rank: task user index out of range");
  *out_n = 0;
  if (out_order_n) *out_order_n = 0;
  if (N == 0) return COOK_OK;
  CK(pool, cudaSetDevice(pool->device));
  cudaStream_t st = pool->stream;
  Arena& ar = pool->arena;
  Sizer sz;
  for (int k = 0; k < 2; k++) sz.add<int32_t>(N + 1);
  for (int k = 0; k < 3; k++) sz.add<int64_t>(N + 1);
  for (int k = 0; k < 3; k++) sz.add<double>(N + 1);
  sz.add<int32_t>(U);
  for (int k = 0; k < 7; k++) sz.add<double>(U);
  for (int k = 0; k < 6; k++) sz.add<int32_t>(N + 1);  // idx,tmp,user_at,pos,out_order,out_ranked
  sz.add<double>(N + 1);                                 // dru_at
  for (int k = 0; k < 2; k++) sz.add<int32_t>(U);        // seg bounds
  sz.add<double>(8);
  sz.add<int32_t>(8);
  sz.add<double>(N + 1);                                 // dru by task (output)
  for (int k = 0; k < 3; k++) sz.add<double>(N + 1);     // queue-order requests
  sz.add<int32_t>(N + 1); sz.add<uint8_t>(N + 1);        // queue-order task index, flags
  sz.add<int32_t>(N / QF_TB + 2); sz.add<GridFlag>(1);
  for (int k = 0; k < 3; k++) sz.add<double>(N + 1);     // order-wide scans: tile-local sums
  sz.add<double>(3 * (N / OS_TILE + 2)); sz.add<int32_t>(N + 1); sz.add<int32_t>(N / OS_TILE + 2);
  sz.add<int32_t>(N + 1); sz.add<int32_t>(N / RS_TB + 2);  // run starts of equal dru, tile maxima
  CK(pool, ar.reserve(sz.off + 4096));
  ar.reset();

  CK(pool, cudaEventRecord(pool->ev[8], st));
  TaskCols t;
  int32_t *d_user, *d_prio; int64_t *d_start, *d_tid, *d_jid; double *d_cpus, *d_mem, *d_gpus;
  CK(pool, upload2(ar, st, running->user, R, pending->user, J, &d_user));
  CK(pool, upload2(ar, st, running->priority, R, pending->priority, J, &d_prio));
  CK(pool, upload2(ar, st, running->start_time, R, pending->start_time, J, &d_start));
  CK(pool, upload2(ar, st, running->task_id, R, pending->task_id, J, &d_tid));
  CK(pool, upload2(ar, st, running->job_id, R, pending->job_id, J, &d_jid));
  CK(pool, upload2(ar, st, running->cpus, R, pending->cpus, J, &d_cpus));
  CK(pool, upload2(ar, st, running->mem, R, pending->mem, J, &d_mem));
  CK(pool, upload2(ar, st, running->gpus, R, pending->gpus, J, &d_gpus));
  t = TaskCols{d_user, d_prio, d_start, d_tid, d_jid, d_cpus, d_mem, d_gpus};
  int32_t* d_name_rank;
  UserCols uc;
  double *dm, *dc, *dg, *qn, *qc, *qm, *qg;
  CK(pool, upload(ar, st, users->name_rank, U, &d_name_rank));
  CK(pool, upload(ar, st, users->div_mem, U, &dm));
  CK(pool, upload(ar, st, users->div_cpus, U, &dc));
  CK(pool, upload(ar, st, users->div_gpus, U, &dg));
  CK(pool, upload(ar, st, users->quota_count, U, &qn));
  CK(pool, upload(ar, st, users->quota_cpus, U, &qc));
  CK(pool, upload(ar, st, users->quota_mem, U, &qm));
  CK(pool, upload(ar, st, users->quota_gpus, U, &qg));
  uc = UserCols{dm, dc, dg, qn, qc, qm, qg};

  int32_t* d_idx = ar.take<int32_t>(N + 1);
  int32_t* d_tmp = ar.take<int32_t>(N + 1);
  int32_t* d_user_at = ar.take<int32_t>(N + 1);
  int32_t* d_pos = ar.take<int32_t>(N + 1);
  int32_t* d_out_order = ar.take<int32_t>(N + 1);
  int32_t* d_out_ranked = ar.take<int32_t>(N + 1);
  double* d_dru_at = ar.take<double>(N + 1);
  int32_t* d_seg_start = ar.take<int32_t>(U);
  int32_t* d_seg_end = ar.take<int32_t>(U);
  double* d_pool_usage = ar.take<double>(8);
  int32_t* d_counters = ar.take<int32_t>(8);  // [0]=n_kept [1]=n_out
  double* d_dru_task = ar.take<double>(N + 1);
  if (!d_dru_task) return set_err(pool, COOK_E_OOM, "cook_rank: arena exhausted");

  GridFlag* d_gf = ar.take<GridFlag>(1);
  const int os_nb = (N + OS_TILE - 1) / OS_TILE;
  double* d_os_pm = ar.take<double>(N + 1); double* d_os_pc = ar.take<double>(N + 1); double* d_os_pg = ar.take<double>(N + 1);
  double* d_os_b = ar.take<double>(3 * (os_nb + 1));
  int32_t* d_os_pv = ar.take<int32_t>(N + 1); int32_t* d_os_bv = ar.take<int32_t>(os_nb + 1);
  const int rs_nb = (N + RS_TB - 1) / RS_TB;
  int32_t* d_run_start = ar.take<int32_t>(N + 1); int32_t* d_rs_tile = ar.take<int32_t>(rs_nb + 1);
  if (ar.failed) return set_err(pool, COOK_E_OOM, "cook_rank: arena exhausted");
  CK(pool, cudaMemsetAsync(d_gf, 0, sizeof(GridFlag), st));
  CK(pool, cudaMemsetAsync(d_seg_start, 0, sizeof(int32_t) * U, st));
  CK(pool, cudaMemsetAsync(d_seg_end, 0, sizeof(int32_t) * U, st));
  CK(pool, cudaMemsetAsync(d_counters, 0, sizeof(int32_t) * 8, st));

  CK(pool, cudaEventRecord(pool->ev[9], st));
  const int TB = 256, nb = (N + TB - 1) / TB;
  grid_check_kernel<<<nb, TB, 0, st>>>(d_cpus, d_mem, d_gpus, N, d_gf);
  iota_kernel<<<nb, TB, 0, st>>>(d_idx, N);
  CK(pool, csort::sort_indices(d_idx, d_tmp, N, LessUserTask{t, d_name_rank}, st));
  seg_bounds_kernel<<<nb, TB, 0, st>>>(d_idx, d_user, N, d_seg_start, d_seg_end, d_user_at);
  {
    OrderScan os;
    os.idx = d_idx; os.t = t; os.uc = uc; os.user_at = d_user_at; os.seg_start = d_seg_start;
    os.n = N; os.dru_mode = pool->dru_mode; os.max_over_quota = params->max_over_quota_jobs; os.gf = d_gf;
    os.pm = d_os_pm; os.pc = d_os_pc; os.pg = d_os_pg; os.bm = d_os_b; os.bc = d_os_b + os_nb + 1; os.bg = d_os_b + 2 * (os_nb + 1);
    os.pv = d_os_pv; os.bv = d_os_bv; os.dru_at = d_dru_at; os.n_kept_total = d_counters;
    os_amount_tiles<<<os_nb, OS_TB, 0, st>>>(os);
    os_amount_totals<<<1, 32, 0, st>>>(os, os_nb);
    os_violation_tiles<<<os_nb, OS_TB, 0, st>>>(os);
    os_violation_totals<<<1, 32, 0, st>>>(os, os_nb);
    os_finish<<<(N + OS_TB - 1) / OS_TB, OS_TB, 0, st>>>(os);
    int warps_per_block = 4;
    int blocks = (U + warps_per_block - 1) / warps_per_block;
    user_fold_kernel<<<blocks, warps_per_block * 32, 0, st>>>(
        d_idx, t, uc, d_seg_start, d_seg_end, U, pool->dru_mode, params->max_over_quota_jobs,
        d_dru_at, d_counters, d_gf, N);
  }
  run_start_tiles<<<rs_nb, RS_TB, 0, st>>>(d_dru_at, d_user_at, d_seg_start, N, d_run_start, d_rs_tile);
  run_start_carry<<<1, 1, 0, st>>>(d_rs_tile, rs_nb);
  run_start_fix<<<rs_nb, RS_TB, 0, st>>>(d_run_start, d_rs_tile, N);
  iota_kernel<<<nb, TB, 0, st>>>(d_pos, N);
  CK(pool, csort::sort_indices(d_pos, d_tmp, N,
                               LessMerge{d_dru_at, d_user_at, d_seg_start, d_name_rank, d_run_start}, st));
  QueueFilterArgs qa;
  qa.pos_sorted = d_pos; qa.idx = d_idx; qa.n_kept = d_counters; qa.R = R;
  qa.cpus = d_cpus; qa.mem = d_mem; qa.gpus = d_gpus;
  qa.filter_offensive = params->filter_offensive;
  qa.off_mem = params->offensive_max_mem_mb; qa.off_cpus = params->offensive_max_cpus;
  qa.out_order = d_out_order; qa.out_ranked = d_out_ranked; qa.out_n = d_counters + 1;
  qa.ti_at = ar.take<int32_t>(N + 1); qa.flag = ar.take<uint8_t>(N + 1);
  qa.xc = ar.take<double>(N + 1); qa.xm = ar.take<double>(N + 1); qa.xg = ar.take<double>(N + 1);
  const int qnb = (N + QF_TB - 1) / QF_TB;
  qa.blk_cnt = ar.take<int32_t>(qnb + 1);
  if (!qa.blk_cnt) return set_err(pool, COOK_E_OOM, "cook_rank: arena exhausted");
  qf_gather_kernel<<<qnb, QF_TB, 0, st>>>(qa);
  if (pool_quota && pool_quota->enabled) {
    pool_usage_kernel<<<1, 32, 0, st>>>(d_cpus, d_mem, d_gpus, R, d_pool_usage, d_gf);
    qf_quota_kernel<<<1, QF_CH, 0, st>>>(qa, *pool_quota, d_pool_usage, d_gf);
  }
  if (group_quota && group_usage && group_quota->enabled) {
    CK(pool, cudaMemcpyAsync(d_pool_usage + 4, group_usage, sizeof(double) * 4, cudaMemcpyHostToDevice, st));
    qf_quota_kernel<<<1, QF_CH, 0, st>>>(qa, *group_quota, d_pool_usage + 4, d_gf);
  }
  qf_count_kernel<<<qnb, QF_TB, 0, st>>>(qa);
  qf_scan_kernel<<<1, 1024, 0, st>>>(qa, qnb);
  qf_scatter_kernel<<<qnb, QF_TB, 0, st>>>(qa);
  if (out_dru) scatter_dru_kernel<<<nb, TB, 0, st>>>(d_idx, d_dru_at, N, d_dru_task);
  CK(pool, cudaGetLastError());
  CK(pool, cudaEventRecord(pool->ev[10], st));
  int32_t h_counters[2] = {0, 0};
  CK(pool, cudaMemcpyAsync(h_counters, d_counters, sizeof(int32_t) * 2, cudaMemcpyDeviceToHost, st));
  CK(pool, cudaStreamSynchronize(st));
  const int32_t n_kept = h_counters[0], n_out = h_counters[1];
  if (n_out > 0)
    CK(pool, cudaMemcpyAsync(out_ranked_idx, d_out_ranked, sizeof(int32_t) * n_out,
                             cudaMemcpyDeviceToHost, st));
  if (out_order && n_kept > 0)
    CK(pool, cudaMemcpyAsync(out_order, d_out_order, sizeof(int32_t) * n_kept,
                             cudaMemcpyDeviceToHost, st));
  if (out_dru) CK(pool, cudaMemcpyAsync(out_dru, d_dru_task, sizeof(double) * N, cudaMemcpyDeviceToHost, st));
  CK(pool, cudaEventRecord(pool->ev[11], st));
  CK(pool, cudaStreamSynchronize(st));
  {
    cook_phase_stats& ps = pool->phase[COOK_PHASE_RANK];
    ps.ms_h2d = ev_ms(pool->ev[8], pool->ev[9]);
    ps.ms_device = ev_ms(pool->ev[9], pool->ev[10]);
    ps.ms_d2h = ev_ms(pool->ev[10], pool->ev[11]);
    ps.h2d_bytes = (int64_t)N * 56 + (int64_t)U * (4 + 7 * 8);   // task columns (56 B per task) + user tables
    ps.d2h_bytes = (int64_t)n_out * 4 + (out_order ? (int64_t)n_kept * 4 : 0) + (out_dru ? (int64_t)N * 8 : 0) + 8;
    int nl = 0;
    for (long long w = csort::TILE; w < N; w <<= 1) nl += 2;   // the two sorts' merge passes
    ps.n_launches = nl + 15;
  }
  *out_n = n_out;
  if (out_order_n) *out_order_n = n_kept;
  return COOK_OK;
}
