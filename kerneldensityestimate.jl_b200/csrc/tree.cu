// tree.cu -- K3: host construction of the reference's tree arrays and the flatten/upload of a
// BallTreeDensity into level-ordered device records.
//
// Behaviour follows (restated, not copied) src/BallTree01.jl:142-173 (most_spread_coord),
// :223-242 (select!), :282-336 (calcStatsBall!), :342-463 (buildBall!/buildTree!/makeBallTree),
// src/BallTreeDensity01.jl:141-231 (calcStatsDensity!, makeBallTreeDensity).  Unlike the
// reference, which swaps every per-leaf array on each partition step, the partition here
// runs on one index permutation and gathers the leaf payload once; node statistics are
// computed afterwards in the recorded post-order.  The resulting arrays are identical.
#include <cfloat>
#include <chrono>
#include <cstdlib>
#include <cmath>
#include <cstring>
#include <limits>
#include <algorithm>
#include <thread>
#include <type_traits>
#include <vector>

#include "gibbs.cuh"

namespace kdeb200 {

namespace {

constexpr int KDEB200_MAX_DIM_HOST = 64;  // the host builder serves any d the reference accepts (the device path: <= 8)

inline double now_ms() {
  return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

// runs fn(begin, end) over [0, n) on up to `threads` host threads (first-touch page faults and gathers of big trees)
template <class F>
void parallel_ranges(int64_t n, int threads, F fn) {
  if (threads <= 1 || n < 65536) {
    fn((int64_t)0, n);
    return;
  }
  std::vector<std::thread> th;
  const int64_t per = (n + threads - 1) / threads;
  for (int t = 1; t < threads; ++t) {
    const int64_t a = t * per, b = (a + per < n) ? a + per : n;
    if (a < b) th.emplace_back([=] { fn(a, b); });
  }
  fn((int64_t)0, per < n ? per : n);
  for (auto &x : th) x.join();
}

struct Builder {
  int d;
  int64_t N;
  const double *pts;          // d x N, original order
  const double *wts_in, *bw_var;
  std::vector<int64_t> ord;   // leaf slot -> original index
  std::vector<double> s_key, s_kq;  // scratch of nth(), indexed by slot
  std::vector<int64_t> s_oq;
  double *centers, *ranges, *wout, *means, *bandwidth;
  int64_t *left, *right, *lowest, *highest, *perm;

  inline double key(int64_t slot, int dim) const { return pts[ord[slot] * d + dim]; }

  // most_spread_coord (src/BallTree01.jl:142-173): slots lo..hi-1 (the last leaf is excluded, as in the reference).
  // The sums keep the reference's order (sequential per dimension), but all d dimensions share ONE pass over the points
  // for the means and one for the variances -- a point's coordinates sit in one cache line, and the 2 d separate passes
  // of the literal form were the cache misses that dominated the top of the tree.
  int spread_dim(int64_t lo, int64_t hi) const {
    const double w = 1.0 / (double)(hi - lo);
    double mean[KDEB200_MAX_DIM_HOST], var[KDEB200_MAX_DIM_HOST];
    for (int k = 0; k < d; ++k) mean[k] = var[k] = 0.0;
    for (int64_t s = lo; s < hi; ++s) {
      const double *x = pts + ord[s] * d;
      for (int k = 0; k < d; ++k) mean[k] = mean[k] + w * x[k];
    }
    for (int64_t s = lo; s < hi; ++s) {
      const double *x = pts + ord[s] * d;
      for (int k = 0; k < d; ++k) {
        const double df = x[k] - mean[k];
        var[k] += df * df;
      }
    }
    double best = 0.0;
    int arg = 0;
    for (int k = 0; k < d; ++k)
      if (var[k] > best) {
        best = var[k];
        arg = k;
      }
    return arg;
  }

  // The reference's quick-select (select!, src/BallTree01.jl:223-242) -- same result, element for element, without its
  // memory behaviour.  One pass of select! over slots [lo, hi] with the pivot in slot lo is a Lomuto partition:
  //   m = lo; for i in lo..hi: if key(i) - key(lo) < 0 { ++m; swap(m, i) };  swap(lo, m)
  // Slots lo+1..m collect the "less" elements in the order they are met; slots m+1..i-1 hold the others as a QUEUE:
  // every less element that arrives sends the queue's front to its back (the swap), every other element joins the back.
  // So the pass is reproduced by streaming the keys once (contiguous copies of the keys of this dimension, no indirect
  // loads), settling the less elements in place and running the queue in a ring buffer -- branch-free, the comparison is
  // a coin flip -- and writing the queue back behind the pivot: L_c, L_1..L_{c-1}, pivot, queue (the final swap moves
  // the last less element to the front and the pivot behind the less block).
  void nth(int dim, int64_t pos, int64_t lo, int64_t hi) {
    const int64_t n0 = hi - lo + 1;
    if (n0 < 2) return;
    if (n0 < 48) {  // tiny ranges: the literal in-place form is cheapest
      nth_inplace(dim, pos, lo, hi);
      return;
    }
    // scratch indexed by slot: concurrent subtrees own disjoint slot ranges, so one set of arrays serves all threads
    double *K = s_key.data(), *kq = s_kq.data() + lo;
    int64_t *oq = s_oq.data() + lo;
    for (int64_t i = lo; i <= hi; ++i) K[i] = pts[ord[i] * d + dim];
    while (lo < hi) {
      const int64_t n = hi - lo + 1;
      if (n < 48) {
        nth_inplace_keys(K, pos, lo, hi);
        return;
      }
      const int64_t r = (lo + hi) / 2;
      std::swap(ord[r], ord[lo]);
      std::swap(K[r], K[lo]);
      const double pk = K[lo];
      const int64_t po = ord[lo];
      int64_t c = 0, qh = 0, qn = 0;  // less count; queue head / size in a ring of capacity n (the queue holds <= n - 1)
      const int64_t cap = n;
      int64_t *O = ord.data();
      for (int64_t i = lo + 1; i <= hi; ++i) {  // i = lo is the pivot itself: pk - pk < 0 is false and m stays lo
        const double kv = K[i];
        const int64_t ov = O[i];
        const int64_t less = (kv - pk < 0.0) ? 1 : 0;
        K[lo + 1 + c] = kv;  // less elements settle in place, in the order they are met (lo + 1 + c <= i: already read);
        O[lo + 1 + c] = ov;  // the slot is simply rewritten by the next candidate when this one is not less
        c += less;
        int64_t tail = qh + qn;
        tail -= (tail >= cap) ? cap : 0;
        // less: the front goes to the back (a no-op write into a free slot while the queue is empty); else: append
        kq[tail] = less ? kq[qh] : kv;
        oq[tail] = less ? oq[qh] : ov;
        const int64_t adv = less & (qn > 0 ? 1 : 0);
        qh += adv;
        qh -= (qh >= cap) ? cap : 0;
        qn += 1 - less;
      }
      const int64_t m = lo + c;
      if (c > 0) {  // the final swap(lo, m): the last less element to the front, the pivot behind the less block
        K[lo] = K[m];
        O[lo] = O[m];
      }
      K[m] = pk;
      O[m] = po;
      const int64_t first = (qn < cap - qh) ? qn : cap - qh;  // the ring in at most two pieces
      std::memcpy(K + m + 1, kq + qh, sizeof(double) * (size_t)first);
      std::memcpy(O + m + 1, oq + qh, sizeof(int64_t) * (size_t)first);
      std::memcpy(K + m + 1 + first, kq, sizeof(double) * (size_t)(qn - first));
      std::memcpy(O + m + 1 + first, oq, sizeof(int64_t) * (size_t)(qn - first));
      if (m <= pos) lo = m + 1;
      if (m >= pos) hi = m - 1;
    }
  }

  void nth_inplace_keys(double *K, int64_t pos, int64_t lo, int64_t hi) {  // select! on the contiguous keys
    while (lo < hi) {
      const int64_t r = (lo + hi) / 2;
      std::swap(ord[r], ord[lo]);
      std::swap(K[r], K[lo]);
      int64_t m = lo;
      const int64_t l0 = lo, h0 = hi;
      for (int64_t i = l0; i <= h0; ++i) {
        if (K[i] - K[l0] < 0.0) {
          ++m;
          std::swap(ord[m], ord[i]);
          std::swap(K[m], K[i]);
        }
      }
      std::swap(ord[lo], ord[m]);
      std::swap(K[lo], K[m]);
      if (m <= pos) lo = m + 1;
      if (m >= pos) hi = m - 1;
    }
  }

  void nth_inplace(int dim, int64_t pos, int64_t lo, int64_t hi) {  // the reference's quick-select, swap for swap
    while (lo < hi) {
      const int64_t r = (lo + hi) / 2;
      std::swap(ord[r], ord[lo]);
      int64_t m = lo;
      const int64_t l0 = lo, h0 = hi;
      for (int64_t i = l0; i <= h0; ++i) {
        // the pivot sits in slot l0 for the whole pass: only slots > l0 are swap targets
        if (key(i, dim) - key(l0, dim) < 0.0) {
          ++m;
          std::swap(ord[m], ord[i]);
        }
      }
      std::swap(ord[lo], ord[m]);
      if (m <= pos) lo = m + 1;
      if (m >= pos) hi = m - 1;
    }
  }

  // leaf payload of slot s (its final occupant is known once the recursion reaches it)
  inline void gather_leaf(int64_t s) {
    const int64_t o = ord[s], node = N + s;
    perm[node] = o + 1;
    wout[node] = wts_in[o];
    for (int k = 0; k < d; ++k) {
      centers[node * d + k] = pts[o * d + k];
      means[node * d + k] = pts[o * d + k];
      bandwidth[node * d + k] = bw_var[k];
      ranges[node * d + k] = 0.0;
    }
  }

  // calcStatsBall! + calcStatsDensity! of one internal node, children done (src/BallTree01.jl:282-336,
  // src/BallTreeDensity01.jl:141-187); single: the one-point tree, whose only child is counted once
  inline void stats(int64_t root, bool single) {
    const int64_t L = left[root - 1];
    const int64_t R = single ? L : right[root - 1];
    double *c = centers + (root - 1) * d, *rg = ranges + (root - 1) * d;
    const double *cl = centers + (L - 1) * d, *cr = centers + (R - 1) * d;
    const double *rl = ranges + (L - 1) * d, *rr = ranges + (R - 1) * d;
    for (int k = 0; k < d; ++k) {
      const double hiL = cl[k] + rl[k], hiR = cr[k] + rr[k];
      const double maxi = hiL > hiR ? hiL : hiR;
      const double loL = cl[k] - rl[k], loR = cr[k] - rr[k];
      const double mini = loL < loR ? loL : loR;
      const double half = (maxi - mini) / 2.0;
      rg[k] = half;
      c[k] = mini + half;
    }
    wout[root - 1] = (L != R) ? wout[L - 1] + wout[R - 1] : wout[L - 1];
    double wl = wout[L - 1], wr = wout[R - 1];
    const double wt = wl + wr + DBL_EPSILON;
    wl /= wt;
    wr /= wt;
    double *m = means + (root - 1) * d, *bwd = bandwidth + (root - 1) * d;
    const double *ml = means + (L - 1) * d, *mr = means + (R - 1) * d;
    const double *bl = bandwidth + (L - 1) * d, *br = bandwidth + (R - 1) * d;
    for (int k = 0; k < d; ++k) {
      const double mk = wl * ml[k] + wr * mr[k];
      m[k] = mk;
      bwd[k] = wl * (bl[k] + ml[k] * ml[k]) + wr * (br[k] + mr[k] * mr[k]) - mk * mk;
    }
  }

  // node ids are the reference's 1-based ids; slots are 0-based leaf positions (node = N+1+slot).
  // The reference hands out internal ids from a running counter in depth-first order (src/BallTree01.jl:415-434);
  // a subtree over n >= 2 leaves consumes exactly n - 2 of them below its root, so the first free id of every
  // subtree is known up front (next0) and disjoint subtrees can be built by different host threads -- topology, leaf
  // payload and node statistics (children before parents) all inside the same recursion.
  void topo(int64_t lo, int64_t hi, int64_t root, int64_t next0, int par_depth) {
    const int64_t nlo = N + 1 + lo, nhi = N + 1 + hi;
    if (lo == hi) {  // single-point tree
      lowest[root - 1] = nlo;
      highest[root - 1] = nhi;
      left[root - 1] = nlo;
      right[root - 1] = -1;
      gather_leaf(lo);
      stats(root, true);
      return;
    }
    const bool tr = (hi - lo + 1 >= 400000) && getenv("KDEB200_TRACE") != nullptr;
    const double t0 = tr ? now_ms() : 0.0;
    const int dim = spread_dim(lo, hi);
    const double t1 = tr ? now_ms() : 0.0;
    const int64_t split = (lo + hi) / 2;
    nth(dim, split, lo, hi);
    if (tr) fprintf(stderr, "[kdeb200]   node of %lld leaves: spread %.1f ms, select %.1f ms\n", (long long)(hi - lo + 1), t1 - t0, now_ms() - t1);
    int64_t l, r, nxt = next0;
    if (split <= lo) l = nlo; else l = nxt++;
    if (split + 1 >= hi) r = nhi; else r = nxt++;
    lowest[root - 1] = nlo;
    highest[root - 1] = nhi;
    left[root - 1] = l;
    right[root - 1] = r;
    const int64_t nleft = split - lo + 1;
    const int64_t next_right = nxt + (nleft >= 2 ? nleft - 2 : 0);
    if (par_depth > 0 && hi - lo + 1 >= 32768 && l != nlo && r != nhi) {
      std::thread th([&] { topo(lo, split, l, nxt, par_depth - 1); });
      topo(split + 1, hi, r, next_right, par_depth - 1);
      th.join();
    } else {
      if (l != nlo) topo(lo, split, l, nxt, 0); else gather_leaf(lo);
      if (r != nhi) topo(split + 1, hi, r, next_right, 0); else gather_leaf(hi);
    }
    stats(root, false);
  }
};

}  // namespace

int tree_build_host(int d, int64_t N, const double *points, const double *weights, const double *bw_var,
                    double *centers, double *ranges, double *wout, double *means, double *bandwidth,
                    int64_t *left, int64_t *right, int64_t *lowest, int64_t *highest, int64_t *perm) {
  if (d < 1 || N < 1) KDE_FAIL(2, "tree_build: need d >= 1 and N >= 1 (got d=%d N=%lld)", d, (long long)N);
  if (d > KDEB200_MAX_DIM_HOST) KDE_FAIL(3, "tree_build: d=%d above %d", d, KDEB200_MAX_DIM_HOST);
  const int64_t NN = 2 * N;
  const double t_0 = now_ms();
  int par_depth = 4;  // up to 16 host threads on large inputs; KDEB200_BUILD_PAR_DEPTH=0 builds on the calling thread
  if (const char *e = getenv("KDEB200_BUILD_PAR_DEPTH")) par_depth = atoi(e);
  const int nthreads = par_depth > 0 ? (int)std::min<unsigned>(1u << par_depth, std::max(1u, std::thread::hardware_concurrency())) : 1;
  Builder b;
  b.d = d; b.N = N; b.pts = points; b.wts_in = weights; b.bw_var = bw_var;
  b.centers = centers; b.ranges = ranges; b.wout = wout; b.means = means; b.bandwidth = bandwidth;
  b.left = left; b.right = right; b.lowest = lowest; b.highest = highest; b.perm = perm;
  b.ord.resize(N);
  if (N >= 48) {
    b.s_key.resize(N); b.s_kq.resize(N);
    b.s_oq.resize(N);
  }
  // Every entry of the outputs is written exactly once: internal nodes 1..N-1 and leaves N+1..2N by the recursion, the
  // index arrays and the unused slot N here (the reference: zeros(...) / ones(Int, 2Np)).  The caller's arrays are
  // usually fresh pages, so the first touch is spread over the threads.
  parallel_ranges(N, nthreads, [&](int64_t a, int64_t e) {
    for (int64_t i = a; i < e; ++i) {
      b.ord[i] = i;
      left[i] = right[i] = lowest[i] = highest[i] = 1;  // internal entries: overwritten for 1..N-1, slot N keeps ones
      perm[i] = 0;
      const int64_t j = N + i;  // leaves
      lowest[j] = highest[j] = left[j] = j + 1;
      right[j] = -1;
    }
  });
  for (int k = 0; k < d; ++k) {
    const int64_t u = (N - 1) * d + k;
    centers[u] = ranges[u] = means[u] = bandwidth[u] = 0.0;
  }
  wout[N - 1] = 0.0;
  const bool trace = getenv("KDEB200_TRACE") != nullptr;
  const double t_a = now_ms();
  b.topo(0, N - 1, 1, 2, par_depth);
  if (trace)
    fprintf(stderr, "[kdeb200] tree_build_host d=%d N=%lld: init %.1f ms, topology + payload + statistics %.1f ms\n", d, (long long)N,
            t_a - t_0, now_ms() - t_a);
  return 0;
}

// ---------------------------------------------------------------- flatten + upload -------
static inline int even_up(int x) { return (x + 1) & ~1; }

int tree_create(int d, int64_t N, const double *means, const double *bandwidth, const double *weights,
                const int64_t *left, const int64_t *right, const int64_t *perm, bool gibbs_records,
                kdeb200_tree_t *out) {
  if (int rc = ensure_init()) return rc;
  if (!out) KDE_FAIL(2, "tree_create: out is NULL");
  if (d < 1 || d > KDEB200_MAX_DIM) KDE_FAIL(3, "tree_create: d=%d outside 1..%d (no CPU fallback)", d, KDEB200_MAX_DIM);
  if (N < 1) KDE_FAIL(3, "tree_create: N must be >= 1");
  if (2 * N >= (int64_t)std::numeric_limits<int32_t>::max()) KDE_FAIL(3, "tree_create: N too large");
  kdeb200_tree_s *t = new kdeb200_tree_s();
  t->d = d;
  t->N = N;
  t->SA = even_up(d + 1);
  t->SC = even_up(2 * d + 1);
  t->SE = even_up(d + 1);
  const int64_t NN = 2 * N;
  auto valid = [&](int64_t i) { return 0 < i && i <= NN; };

  // uniform leaf bandwidth is what the typed constructors of the reference always produce
  for (int k = 0; k < d; ++k) t->hvar[k] = bandwidth[N * d + k];
  for (int k = 0; k < d; ++k) t->root_mean[k] = means[k];
  for (int k = 0; k < d; ++k) t->root_var[k] = bandwidth[k];
  for (int64_t i = N; i < NN; ++i)
    for (int k = 0; k < d; ++k)
      if (bandwidth[i * d + k] != t->hvar[k] && !(std::isnan(bandwidth[i * d + k]) && std::isnan(t->hvar[k]))) {
        delete t;
        KDE_FAIL(4, "tree_create: per-point bandwidths (multibandwidth != 0) are not supported");
      }

  // BFS level lists exactly as levelDown! produces them (left then right, leaves persist); an
  // evaluation-only tree (kdeb200_tree_create_eval) carries the leaf records alone
  std::vector<std::vector<int64_t>> lists;
  if (gibbs_records) lists.push_back({1});
  while (gibbs_records) {
    const std::vector<int64_t> &cur = lists.back();
    std::vector<int64_t> nxt;
    nxt.reserve(cur.size() * 2);
    for (int64_t y : cur) {
      const int64_t l = left[y - 1], r = right[y - 1];
      if (valid(l)) nxt.push_back(l);
      if (valid(r)) nxt.push_back(r);
    }
    if (nxt == cur) break;
    if ((int64_t)nxt.size() > N || lists.size() > 80) {
      delete t;
      KDE_FAIL(4, "tree_create: malformed child arrays (level list exceeds N)");
    }
    lists.push_back(std::move(nxt));
  }
  t->gibbs_ready = gibbs_records;
  t->depth = gibbs_records ? (int)lists.size() - 1 : 0;
  if (gibbs_records)
  for (int64_t y : lists.back())
    if (y <= N) {
      delete t;
      KDE_FAIL(4, "tree_create: malformed tree (internal node %lld without children)", (long long)y);
    }

  // lay the records out
  t->levels.resize(lists.size());
  int64_t off = 0;
  auto take = [&](int64_t n) { int64_t o = off; off += (n + 1) & ~(int64_t)1; return o; };
  for (size_t l = 0; l < lists.size(); ++l) {
    kdeb200::Level &L = t->levels[l];
    L.n = (int64_t)lists[l].size();
    bool all_leaf = true;
    for (int64_t y : lists[l]) all_leaf = all_leaf && (y > N);
    L.cls = (all_leaf && l > 0) ? 0 : 1;
    L.offW = take(L.n);
    if (L.cls == 0) {
      L.offA = take(L.n * t->SA);
    } else {
      L.offB = take(L.n * t->SC);
      L.offC = take(L.n * t->SC);
    }
  }
  t->buf_doubles = (size_t)off;
  std::vector<double> h(off, 0.0);
  bool degen = false;
  for (size_t l = 0; l < lists.size(); ++l) {
    const kdeb200::Level &L = t->levels[l];
    for (int64_t z = 0; z < L.n; ++z) {
      const int64_t y = lists[l][z];
      const double w = weights[y - 1];
      const double lw = std::log(w);
      h[L.offW + z] = w;
      if (!(w >= 0.0) || !std::isfinite(w)) degen = true;
      if (L.cls == 0) {
        double *r = &h[L.offA + z * t->SA];
        for (int k = 0; k < d; ++k) {
          r[k] = means[(y - 1) * d + k];
          if (!std::isfinite(r[k])) degen = true;
        }
        r[d] = lw;
      } else {
        double *rb = &h[L.offB + z * t->SC], *rc = &h[L.offC + z * t->SC];
        double sl = 0.0;
        for (int k = 0; k < d; ++k) {
          const double m = means[(y - 1) * d + k], b = bandwidth[(y - 1) * d + k];
          if (!std::isfinite(m) || !std::isfinite(b) || !(b > 0.0)) degen = true;
          rb[k] = rc[k] = m;
          rb[d + k] = -0.5 / b;
          rc[d + k] = b;
          sl += std::log(b);
        }
        rb[2 * d] = lw - 0.5 * sl;
        rc[2 * d] = lw;
      }
    }
  }
  for (int k = 0; k < d; ++k)
    if (!(t->hvar[k] > 0.0) || !std::isfinite(t->hvar[k])) degen = true;
  // Range contract of the fast arithmetic (kde_exp_flush needs exponents <= 700, the one-rsqrt normaliser needs
  // prod_k c_k to stay normal at d = 8): every variance in [1e-30, 1e30], every mean within 1e100.  Anything
  // outside is refused by the Gibbs entry points (code 8) instead of producing a wrong CDF.
  auto var_ok = [](double b) { return b >= 1e-30 && b <= 1e30; };
  for (int k = 0; k < d; ++k)
    if (!var_ok(t->hvar[k])) degen = true;
  if (gibbs_records)
    for (int64_t i = 0; i + 1 < N && !degen; ++i)
      for (int k = 0; k < d; ++k)
        if (!var_ok(bandwidth[i * d + k]) || !(std::fabs(means[i * d + k]) <= 1e100)) degen = true;
  t->degenerate = degen;

  // leaf-order evaluation records and labels
  std::vector<double> leaf((size_t)N * t->SE, 0.0);
  std::vector<int64_t> pr(N), lab(gibbs_records ? lists.back().size() : 0);
  for (int64_t s = 0; s < N; ++s) {
    const int64_t node = N + s;
    for (int k = 0; k < d; ++k) {
      const double x = means[node * d + k];
      leaf[s * t->SE + k] = x;
      const double dev = std::fabs(x - t->root_mean[k]);
      if (dev > t->extent[k] || dev != dev) t->extent[k] = dev;
    }
    leaf[s * t->SE + d] = weights[node];
    pr[s] = perm[node] - 1;
    if (pr[s] < 0 || pr[s] >= N) {
      delete t;
      KDE_FAIL(4, "tree_create: permutation entry out of range at leaf %lld", (long long)s);
    }
  }
  for (size_t z = 0; z < lab.size(); ++z) lab[z] = perm[lists.back()[z] - 1] + 1;
  std::vector<int64_t> levperm;
  for (size_t l = 0; l < lists.size(); ++l) {
    t->levels[l].offP = (int64_t)levperm.size();
    for (int64_t y : lists[l]) levperm.push_back(perm[y - 1]);
  }

  // one stream-ordered allocation for everything (cudaFree of five blocks cost 33 ms per tree)
  Context &c = ctx();
  auto up = [](size_t b) { return (b + 255) & ~(size_t)255; };
  const size_t b_rec = up(sizeof(double) * h.size()), b_lab = up(sizeof(int64_t) * lab.size()),
               b_lp = up(sizeof(int64_t) * levperm.size()), b_leaf = up(sizeof(double) * leaf.size()),
               b_perm = up(sizeof(int64_t) * pr.size());
  const size_t total = b_rec + b_lab + b_lp + b_leaf + b_perm;
  char *base = nullptr;
  cudaError_t e = cudaMallocAsync(&base, total, c.stream);
  if (e != cudaSuccess) {
    set_error("tree_create: cudaMallocAsync(%zu bytes): %s", total, cudaGetErrorString(e));
    delete t;
    return 100 + (int)e;
  }
  t->d_base = base;
  t->d_buf = reinterpret_cast<double *>(base);
  t->d_labels = reinterpret_cast<int64_t *>(base + b_rec);
  t->d_levperm = reinterpret_cast<int64_t *>(base + b_rec + b_lab);
  t->d_leaf = reinterpret_cast<double *>(base + b_rec + b_lab + b_lp);
  t->d_perm = reinterpret_cast<int64_t *>(base + b_rec + b_lab + b_lp + b_leaf);
  auto fail = [&](cudaError_t err, const char *what) {
    set_error("tree_create: %s: %s", what, cudaGetErrorString(err));
    cudaFreeAsync(base, c.stream);
    delete t;
    return 100 + (int)err;
  };
  if ((e = cudaMemcpyAsync(t->d_buf, h.data(), sizeof(double) * h.size(), cudaMemcpyHostToDevice, c.stream)) != cudaSuccess) return fail(e, "H2D records");
  if ((e = cudaMemcpyAsync(t->d_labels, lab.data(), sizeof(int64_t) * lab.size(), cudaMemcpyHostToDevice, c.stream)) != cudaSuccess) return fail(e, "H2D labels");
  if ((e = cudaMemcpyAsync(t->d_levperm, levperm.data(), sizeof(int64_t) * levperm.size(), cudaMemcpyHostToDevice, c.stream)) != cudaSuccess) return fail(e, "H2D levperm");
  if ((e = cudaMemcpyAsync(t->d_leaf, leaf.data(), sizeof(double) * leaf.size(), cudaMemcpyHostToDevice, c.stream)) != cudaSuccess) return fail(e, "H2D leaves");
  if ((e = cudaMemcpyAsync(t->d_perm, pr.data(), sizeof(int64_t) * pr.size(), cudaMemcpyHostToDevice, c.stream)) != cudaSuccess) return fail(e, "H2D perm");
  if ((e = cudaStreamSynchronize(c.stream)) != cudaSuccess) return fail(e, "sync");  // host vectors die here
  t->device_bytes = total;
  t->slot = c.slot;
  t->device = c.device;
  t->h_perm = std::move(pr);
  *out = t;
  return 0;
}

// Replica of a tree on another GPU of the in-process set: ONE peer copy of the single allocation (NVLink when peer
// access is on, staged by the driver otherwise), every pointer rebased.  Created on first use, freed with the tree.
int tree_on(kdeb200_tree_t t, int slot, kdeb200_tree_t *out) {
  if (!t) KDE_FAIL(2, "tree_on: NULL tree");
  if (slot == t->slot) {
    *out = t;
    return 0;
  }
  if (t->slot != 0) KDE_FAIL(3, "tree_on: only trees created on the primary device can be replicated");
  if (slot < 0 || slot >= multi_count()) KDE_FAIL(3, "tree_on: slot %d outside the multi-GPU set", slot);
  if (t->replica[slot] && t->replica[slot]->device == ctx_at(slot).device) {
    *out = t->replica[slot];
    return 0;
  }
  // (a replica made for another device list -- kdeb200_init_multi_devices was called again -- is left to its pool)
  Context &src = ctx_at(0);
  Context &dst = ctx_at(slot);
  ScopedDevice sd(slot);
  char *base = nullptr;
  KDE_CUDA(cudaMallocAsync(&base, t->device_bytes, dst.stream));
  cudaError_t e = cudaMemcpyPeerAsync(base, dst.device, t->d_base, src.device, t->device_bytes, dst.stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(dst.stream);
  if (e != cudaSuccess) {
    cudaFreeAsync(base, dst.stream);
    KDE_FAIL(100 + (int)e, "tree_on: peer copy to device %d: %s", dst.device, cudaGetErrorString(e));
  }
  kdeb200_tree_s *r = new kdeb200_tree_s(*t);
  for (auto &p : r->replica) p = nullptr;
  const ptrdiff_t off = base - t->d_base;
  auto rebase = [&](auto *&p) {
    if (p) p = reinterpret_cast<std::remove_reference_t<decltype(p)>>(reinterpret_cast<char *>(p) + off);
  };
  r->d_base = base;
  rebase(r->d_buf);
  rebase(r->d_labels);
  rebase(r->d_levperm);
  rebase(r->d_leaf);
  rebase(r->d_perm);
  r->device = dst.device;
  r->d_leaf32 = nullptr;
  r->d_tilebox = nullptr;
  r->d_tilebox32 = nullptr;
  r->d_cw = nullptr;
  r->d_leaf_of = nullptr;
  r->slot = slot;
  t->replica[slot] = r;
  *out = r;
  return 0;
}

int tree_destroy(kdeb200_tree_t t) {
  if (!t) return 0;
  if (t->gibbs_ready) gibbs_invalidate_schedules();
  // Kernels of the *_device entry points may still be running on a caller stream: drain the device (microseconds
  // when idle), then release with the stream-ordered allocator (cudaFree cost 33 ms per tree).
  Context &c = ctx();
  const bool trace = getenv("KDEB200_TRACE") != nullptr;
  auto now = [] { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
  const double t0 = now();
  cudaDeviceSynchronize();
  const double t1 = now();
  if (t->d_base) cudaFreeAsync(t->d_base, c.stream);
  if (t->d_leaf32) cudaFreeAsync(t->d_leaf32, c.stream);
  if (t->d_tilebox) cudaFreeAsync(t->d_tilebox, c.stream);
  if (t->d_tilebox32) cudaFreeAsync(t->d_tilebox32, c.stream);
  if (t->d_cw) cudaFreeAsync(t->d_cw, c.stream);
  for (int s = 1; s < KDEB200_MAX_GPUS; ++s)
    if (kdeb200_tree_s *r = t->replica[s]) {
      if (s < multi_count() && ctx_at(s).ready && ctx_at(s).device == r->device) {  // else: the set was re-made without this device
        ScopedDevice sd(s);
        cudaDeviceSynchronize();
        if (r->d_base) cudaFreeAsync(r->d_base, ctx_at(s).stream);
        if (r->d_leaf32) cudaFreeAsync(r->d_leaf32, ctx_at(s).stream);
        if (r->d_tilebox) cudaFreeAsync(r->d_tilebox, ctx_at(s).stream);
        if (r->d_tilebox32) cudaFreeAsync(r->d_tilebox32, ctx_at(s).stream);
        if (r->d_cw) cudaFreeAsync(r->d_cw, ctx_at(s).stream);
      }
      delete r;
    }
  const double t2 = now();
  delete t;
  if (trace) fprintf(stderr, "[kdeb200] tree_destroy: sync %.3f ms, free %.3f ms, delete %.3f ms\n", t1 - t0, t2 - t1, now() - t2);
  return 0;
}

}  // namespace kdeb200
