// gibbs_exact_kernel.cuh -- K1x (device code and launch template; gibbs_exact.cu holds the host side,
// gibbs_exact_d<N>.cu one explicit instantiation per d): the FP64 Gibbs sampler with the labels of the leaf levels
// DECIDED from certified FP32 prefix sums.
//
// Same schedule, chain state, RNG addressing and outputs as gibbs_kernel (K1), bit for bit.  K1 picks on every level
// the first z with target = fl(u * pT) <= S_z, S_z its sequential FP64 prefix sums (else n - 1).  On the leaf levels
// (variant A, two thirds of K1's FP64 work at C4) K1x instead evaluates the nodes in packed FP32 (gibbs_f32_kernel.cuh's
// pair records and arithmetic) and carries next to every FP32 prefix sum S'_z a bound E_z on |S'_z - S_z / W|
// (W: the level's largest weight; DESIGN.md "K1x" derives it).  A lane's label is taken only when the intervals prove
// it:  hi(S_{z-1}) < lo(target)  and  hi(target) <= lo(S_z).  A lane that cannot prove its label is redone by its
// warp with K1's FP64 arithmetic (K1w's scheme: lanes evaluate, one lane sums in node order, the result is K1's
// label by construction).  Internal levels (variants B, C) run K1's own pass1 / pass2 unchanged.
#pragma once
#include "gibbs_f32_kernel.cuh"

namespace kdeb200 {

constexpr int GX_SCR = 256;  // doubles of global scratch per warp (the cooperative FP64 redo)

// per-draw extras of K1x (variant-A draws only; zero elsewhere)
struct alignas(16) XDraw {
  const float *rec32;                 // FP32 pair records, coordinates relative to the tile centre
  const double *ctr;                  // tile centres, KDEB200_MAX_DIM doubles per tile of this draw
  double rad[KDEB200_MAX_DIM];        // max over the level of |m - centre| per dimension (FP64, rounded up)
  double lw2max;                      // log2 of the level's largest weight (records hold lw2max - log2 w >= 0)
  int G, nchunks;                     // K1x's own checkpoint chunks (nodes, power of two)
  int fp32;                           // 0: the level is outside the FP32 range guard, every lane takes the FP64 redo
  int pad;
};

struct XParams {
  const XDraw *xd;
  double *scratch;                    // GX_SCR doubles per warp of the grid
  unsigned long long *redone;         // lane-draws redone in FP64 (live chains only)
  unsigned long long *warp_redone;    // warp-draws with at least one redone lane
  double ex2_err;                     // relative error bound of ex2.approx.ftz.f32 on [-126, 0]
  double inflate;                     // test hook: multiplies the bound (1 in production)
};

// The bound of one variant-A draw: |p32 - p64 / W| <= p32 (A + B acc32) per node, plus aabs; prefix sums add the
// summation terms.  DESIGN.md "K1x" derives every constant.
struct XBound {
  double A, B, aabs, eta;
  bool ok;
};

template <int D>
__device__ __forceinline__ XBound xa_bound(const XDraw &xd, const float (&s32)[D], int n, double ex2_err, double inflate) {
  const double u = 0x1.0p-24 * (1.0 + 0x1.0p-20);
  double Rmax = 0.0, Rsum = 0.0, R2 = 0.0;
#pragma unroll
  for (int k = 0; k < D; ++k) {
    const double R = xd.rad[k] * (double)s32[k] * (1.0 + 3.0 * u);
    Rmax = fmax(Rmax, R);
    Rsum += R;
    R2 += R * R;
  }
  const double a1 = (D + 7.2) * u + 2.05 * u * Rmax;
  const double a0 = 2.05 * u * Rsum + 1e-13 * R2;
  XBound b;
  b.ok = xd.fp32 && (a1 * 130.0 + a0 <= 1e-3) && (R2 == R2);
  const double ln2 = 0.6931471805599453;
  const double lwm = fabs(xd.lw2max);
  // pass 1 adds Q's terms (non-negative) in FP32 over a whole chunk of G nodes before folding them into FP64: the
  // computed chunk sum is at least (1 - G u) of the exact one, so B carries the factor 1 / (1 - G u)
  const double qsum = 1.0 / (1.0 - (double)xd.G * u);
  b.ok = b.ok && (double)xd.G * u < 0.1;
  b.B = inflate * qsum * (1.003 * ln2 * 1.001 * a1 + 5e-15);
  b.A = inflate * (1.003 * (ln2 * (a0 + 1.001 * a1 * a0) + 1.01 * ex2_err) + 2.0 * gf_unr(D, VAR_A) * 1.01 * u +
                   (double)n * 0x1.0p-52 + 1e-15 * (6.0 + lwm));
  // ex2.approx.ftz flushes 2^-acc below 2^-126 to zero; K1 clamps exponents below -700 (kde_exp_flush)
  b.aabs = 0x1.0p-125 + exp(-699.0 - xd.lw2max * ln2);
  b.eta = (double)n * 1.2e-16 + 1e-15;
  return b;
}

__device__ __forceinline__ double xa_err(const XBound &b, double S, double Q, int cnt) {
  return 1.01 * (b.A * S + b.B * Q) + (double)cnt * b.aabs;
}

// b_k = (mu_k - centre_k) s_k in FP64 once per tile, clamped so that FP32 never sees an infinity
template <int D>
__device__ __forceinline__ void xa_tile_hoist(const double *__restrict__ ctr, const double (&mu)[D], const float (&s32)[D],
                                              Hoist32<D> &g) {
#pragma unroll
  for (int k = 0; k < D; ++k) {
    const double bk = fmin(fmax((mu[k] - ctr[k]) * (double)s32[k], -1e12), 1e12);
    const float fb = (float)(-bk);
    g.b[k] = gf_pack(fb, fb);
  }
}

// pass 1 over the FP32 tiles of a variant-A draw: trip sums of 2 UNR terms in FP32 folded into an FP64 running sum,
// Q = sum p32 acc32 (the exponent-proportional part of the bound), both checkpointed every G nodes
template <int D>
__device__ __forceinline__ double xa_pass1(const Draw &dr, const XDraw &xd, const double (&mu)[D], const float (&s32)[D],
                                           Ring &R, int64_t &q, double *__restrict__ ck, float *__restrict__ ckq, double &Qout) {
  constexpr int UNR = gf_unr(D, VAR_A);
  constexpr int stride = gf_stride(D, VAR_A);
  Hoist32<D> g;
#pragma unroll
  for (int k = 0; k < D; ++k) g.a[k] = gf_pack(s32[k], s32[k]);
  const int npt = (dr.n + 1) >> 1;
  const int Gp = xd.G >> 1;
  const int tp = dr.tnodes >> 1;
  double S = 0.0, Q = 0.0;
  float qf = 0.f;
  int c = 0, done = 0, left = Gp;
  for (int t = 0; t < dr.ntiles; ++t, ++q) {
    xa_tile_hoist<D>(xd.ctr + (size_t)t * KDEB200_MAX_DIM, mu, s32, g);
    const int np = (npt - done < tp) ? (npt - done) : tp;
    mbar_wait(&R.bars[q % GB_STAGES], (uint32_t)((q / GB_STAGES) & 1));
    const float *rec = reinterpret_cast<const float *>(R.tiles + (size_t)(q % GB_STAGES) * (GB_TILE_BYTES / 8));
    int zp = 0;
    while (zp < np) {
      const int run = (left < np - zp) ? left : (np - zp);
      const float *r = rec + (size_t)zp * stride;
      int i = 0;
      for (; i + UNR <= run; i += UNR) {
        f32x2 acc[UNR], sc[UNR];
        gf_trip_pre<D, VAR_A, UNR>(r + (size_t)i * stride, g, acc, sc);
        float s = 0.f;
#pragma unroll
        for (int uu = 0; uu < UNR; ++uu) {
          float al, ah;
          gf_unpack(acc[uu], al, ah);
          const float pa = gf_ex2_neg(al), pb = gf_ex2_neg(ah);
          s = __fadd_rn(s, pa);
          s = __fadd_rn(s, pb);
          qf = __fmaf_rn(pa, al, qf);
          qf = __fmaf_rn(pb, ah, qf);
        }
        S = __dadd_rn(S, (double)s);
      }
      for (; i < run; ++i) {
        f32x2 acc[1], sc[1];
        gf_trip_pre<D, VAR_A, 1>(r + (size_t)i * stride, g, acc, sc);
        float al, ah;
        gf_unpack(acc[0], al, ah);
        const float pa = gf_ex2_neg(al), pb = gf_ex2_neg(ah);
        S = __dadd_rn(S, (double)__fadd_rn(pa, pb));
        qf = __fmaf_rn(pa, al, qf);
        qf = __fmaf_rn(pb, ah, qf);
      }
      zp += run;
      done += run;
      left -= run;
      if (left == 0 || done == npt) {
        Q = __dadd_rn(Q, (double)qf);
        qf = 0.f;
        ck[c] = S;
        ckq[c] = __double2float_ru(Q);
        ++c;
        left = Gp;
      }
    }
    __syncthreads();  // stage free again
    if (threadIdx.x == 0) ring_fill(R, q + 1);
  }
  Qout = Q;
  return S;
}

// decision: chunk from the central checkpoint values, then per-node intervals over that chunk (FP32 terms from global
// memory, FP64 running sums).  Returns the certified label or -1.
template <int D>
__device__ __forceinline__ int xa_decide(const Draw &dr, const XDraw &xd, const XBound &bd, const double (&mu)[D],
                                         const float (&s32)[D], const double *__restrict__ ck, const float *__restrict__ ckq,
                                         double tc, double tLo, double tHi) {
  constexpr int stride = gf_stride(D, VAR_A);
  const int n = dr.n;
  int lo = 0, hi = xd.nchunks;
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (tc <= ck[mid]) hi = mid; else lo = mid + 1;
  }
  if (lo >= xd.nchunks) lo = xd.nchunks - 1;
  const int z0 = lo * xd.G;
  const int z1 = (z0 + xd.G < n) ? z0 + xd.G : n;
  double S = 0.0, Q = 0.0, prevHi = 0.0;
  if (lo > 0) {
    S = ck[lo - 1];
    Q = (double)ckq[lo - 1];
    prevHi = (S + xa_err(bd, S, Q, z0)) * (1.0 + bd.eta);
  }
  Hoist32<D> g;
#pragma unroll
  for (int k = 0; k < D; ++k) g.a[k] = gf_pack(s32[k], s32[k]);
  int cur = -1;
  for (int z = z0; z < z1; z += 2) {
    const int t = z / dr.tnodes;
    if (t != cur) {
      xa_tile_hoist<D>(xd.ctr + (size_t)t * KDEB200_MAX_DIM, mu, s32, g);
      cur = t;
    }
    f32x2 acc, sc;
    gf_pre<D, VAR_A, true>(xd.rec32 + (size_t)(z >> 1) * stride, g, acc, sc);
    float al, ah;
    gf_unpack(acc, al, ah);
    const float pp[2] = {gf_ex2_neg(al), gf_ex2_neg(ah)};
    const float aa[2] = {al, ah};
#pragma unroll
    for (int hh = 0; hh < 2; ++hh) {
      const int zz = z + hh;
      if (zz >= z1) break;
      S = __dadd_rn(S, (double)pp[hh]);
      Q = __fma_rn((double)pp[hh], (double)aa[hh], Q);
      const double E = xa_err(bd, S, Q, zz + 1);
      const double sLo = (S - E) * (1.0 - bd.eta), sHi = (S + E) * (1.0 + bd.eta);
      if (tHi <= sLo || zz == n - 1) return (zz == 0 || prevHi < tLo) ? zz : -1;
      prevHi = sHi;
    }
  }
  return -1;
}

// K1's label for one lane's variant-A draw, computed by the whole warp: lanes evaluate the nodes with K1's eval_node,
// lane 0 adds them in node order (the same additions as K1's pass 1 and pass 2), pT < 1e-99 rule included.
template <int D>
__device__ __noinline__ int xa_redo(const Draw &dr, const Hoist<D, false> &h, double scale, double u,
                                    const double *__restrict__ tab, const ExpConsts &ec, double *__restrict__ scr) {
  const unsigned FULL = 0xffffffffu;
  const int lane = threadIdx.x & 31;
  const int n = dr.n;
  double S = 0.0;
  for (int base = 0; base < n; base += GX_SCR) {
    const int cnt = (n - base < GX_SCR) ? n - base : GX_SCR;
    for (int i = lane; i < cnt; i += 32) scr[i] = eval_node<D, false, VAR_A, true>(dr.rec + (size_t)(base + i) * dr.stride, h, tab, ec);
    __syncwarp();
    if (lane == 0)
      for (int i = 0; i < cnt; ++i) S = __dadd_rn(S, scr[i]);
    __syncwarp();
  }
  const double pT = __shfl_sync(FULL, S, 0);
  int zs = n - 1;
  if (pT * scale < 1e-99) {  // :311-315: all p[z] = weight(last node)
    if (lane == 0) {
      const double w = dr.wts[n - 1];
      double tot = 0.0;
      for (int z = 0; z < n; ++z) tot += w;
      const double qv = w / tot;
      double cdf = 0.0;
      bool found = false;
      for (int z = 0; z < n - 1; ++z) {
        cdf += qv;
        if (!found && u <= cdf) {
          zs = z;
          found = true;
        }
      }
    }
    return __shfl_sync(FULL, zs, 0);
  }
  const double target = u * pT;
  S = 0.0;
  for (int base = 0; base < n; base += GX_SCR) {
    const int cnt = (n - base < GX_SCR) ? n - base : GX_SCR;
    for (int i = lane; i < cnt; i += 32) scr[i] = eval_node<D, false, VAR_A, true>(dr.rec + (size_t)(base + i) * dr.stride, h, tab, ec);
    __syncwarp();
    int f = -1;
    if (lane == 0)
      for (int i = 0; i < cnt; ++i) {
        S = __dadd_rn(S, scr[i]);
        if (target <= S) {
          f = base + i;
          break;
        }
      }
    f = __shfl_sync(FULL, f, 0);
    __syncwarp();
    if (f >= 0) return f;
  }
  return zs;
}

template <int D, int MD>
__global__ void __launch_bounds__(GB_THREADS, GB_MINBLOCKS) gibbs_exact_kernel(const __grid_constant__ GibbsParams P,
                                                                               const __grid_constant__ XParams X) {
  constexpr bool MASK = false;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  double *tiles = reinterpret_cast<double *>(smem_raw);
  __shared__ __align__(16) double tab[KDE_EXP_TAB];
  __shared__ __align__(8) uint64_t bars[GB_STAGES];
  const int tid = threadIdx.x, lane = tid & 31;
  const int M = P.M;
  const unsigned FULL = 0xffffffffu;
  double *scr = X.scratch + ((size_t)blockIdx.x * (GB_THREADS / 32) + (tid >> 5)) * GX_SCR;

  for (int i = tid; i < KDE_EXP_TAB; i += GB_THREADS) tab[i] = P.exptab[i];
  if (tid == 0) {
    for (int s = 0; s < GB_STAGES; ++s) mbar_init(&bars[s], 1);
    mbar_fence_init();
  }
  __syncthreads();

  // dynamic batch scheduling exactly as in gibbs_kernel
  __shared__ int claim;
  const int last_ticket = P.nbatches + (int)gridDim.x - 1;
  if (tid == 0) {
    claim = atomicAdd(P.counter, 1);
    if (claim == last_ticket) *P.counter = 0;
  }
  __syncthreads();
  int batch = claim, batch_next = P.nbatches;
  Ring R;
  R.tiles = tiles;
  R.bars = bars;
  R.descs = P.tiles;
  R.ntiles = P.ntiles;
  R.known = (batch < P.nbatches) ? P.ntiles : 0;
  R.issued = 0;
  R.nxt = P.tiles[0];
  R.nxt_idx = 0;
  if (tid == 0) ring_fill(R, 0);
  int64_t q = 0;

  double lam[MD * D];
  double lmu[MD * D];
  double ck[GB_MAXCK];
  float ckq[GB_MAXCK];
  int selpos[MD];
  unsigned redone = 0, wredone = 0;

  while (batch < P.nbatches) {
    int64_t s = P.s0 + (int64_t)batch * GB_THREADS + tid;
    const bool live = s < P.s1;
    if (!live) s = P.s1 - 1;  // idle lanes replay the last chain (keeps the CTA in lock-step)

    for (int j = 0; j < M; ++j) {
      const double *rr = P.root_rec[j];
#pragma unroll
      for (int k = 0; k < D; ++k) {
        const double l = 1.0 / rr[D + k];
        lam[j * D + k] = l;
        lmu[j * D + k] = rr[k] * l;
      }
      selpos[j] = 0;
    }

    double X_[D];
    for (int di = 0; di < P.ndraws; ++di) {
      const Draw dr = P.draws[di];
      const int j = dr.j;
      if (di == P.ndraws - 1) {
        __syncthreads();
        if (tid == 0) {
          claim = atomicAdd(P.counter, 1);
          if (claim == last_ticket) *P.counter = 0;
        }
        __syncthreads();
        batch_next = claim;
        if (batch_next < P.nbatches) R.known += P.ntiles;
      }

      if (dr.new_level) {  // samplePoint!(addEntropy = true), K1's expressions
#pragma unroll
        for (int k = 0; k < D; ++k) {
          double Lm = 0.0, Hm = 0.0;
          for (int i = 0; i < M; ++i) {
            Lm += lam[i * D + k];
            Hm += lmu[i * D + k];
          }
          const uint32_t slot = (uint32_t)((dr.level - 1) * D + k);
          const double g = P.randN ? P.randN[s * P.perN + slot] : philox_normal(P.seed, (uint64_t)s, slot);
          const double cov = 1.0 / Lm;
          X_[k] = cov * Hm + sqrt(cov) * g;
        }
      }

      Hoist<D, MASK> h;
      double scale = 1.0;
      if (dr.kind == 0) {
#pragma unroll
        for (int k = 0; k < D; ++k) {
          h.mu[k] = X_[k];
          h.cadd[k] = 0.0;
          h.act[k] = true;
        }
      } else {
#pragma unroll
        for (int k = 0; k < D; ++k) {
          double Lm = 0.0, Hm = 0.0;
          for (int i = 0; i < M; ++i) {
            if (i == j) continue;
            Lm += lam[i * D + k];
            Hm += lmu[i * D + k];
          }
          const double cov = 1.0 / Lm;  // M > 1 on this route
          h.cadd[k] = cov;
          h.mu[k] = cov * Hm;
          h.act[k] = true;
        }
      }
      float s32[D];
      if (dr.variant == VAR_A) {
        double prod = 1.0;
#pragma unroll
        for (int k = 0; k < D; ++k) {
          const double c = P.hvar[j][k] + h.cadd[k];
          h.ich[k] = sqrt(0.5 / c);
          prod *= c;
          s32[k] = (float)sqrt(GF_HL2E / c);
        }
        scale = kde_rsqrt(prod);
      }

      int zs = 0;
      if (dr.variant == VAR_A) {
        const XDraw xd = X.xd[di];
        double Qt;
        const double pT = xa_pass1<D>(dr, xd, h.mu, s32, R, q, ck, ckq, Qt);
        bool und = false;
        double u = 0.0;
        if (dr.n > 1) {
          const uint32_t c = (uint32_t)(M + di);
          u = P.randU ? P.randU[s * P.perU + c - 1] : philox_uniform(P.seed, (uint64_t)s, c);
          const XBound bd = xa_bound<D>(xd, s32, dr.n, X.ex2_err, X.inflate);
          const double E = xa_err(bd, pT, Qt, dr.n);
          const double pLo = (pT - E) * (1.0 - bd.eta), pHi = (pT + E) * (1.0 + bd.eta);
          // K1's pT * scale < 1e-99 rule must provably not fire; u in [0, 1) keeps the target interval ordered
          und = !(bd.ok && u >= 0.0 && u < 1.0 && pLo > 0.0 && pLo * exp2(xd.lw2max) * scale >= 1.000001e-99);
          if (!und) {
            const double tLo = u * pLo * (1.0 - 0x1.0p-50), tHi = u * pHi * (1.0 + 0x1.0p-50);
            zs = xa_decide<D>(dr, xd, bd, h.mu, s32, ck, ckq, u * pT, tLo, tHi);
            und = zs < 0;
          }
        }
        unsigned ub = __ballot_sync(FULL, und);
        if (ub) {
          if (live && und) ++redone;
          if (lane == 0) ++wredone;
        }
        while (ub) {
          const int L = __ffs(ub) - 1;
          ub &= ub - 1;
          Hoist<D, MASK> hl;
#pragma unroll
          for (int k = 0; k < D; ++k) {
            hl.mu[k] = __shfl_sync(FULL, h.mu[k], L);
            hl.ich[k] = __shfl_sync(FULL, h.ich[k], L);
            hl.cadd[k] = 0.0;
            hl.act[k] = true;
          }
          const int zl = xa_redo<D>(dr, hl, __shfl_sync(FULL, scale, L), __shfl_sync(FULL, u, L), tab, P.ec, scr);
          if (lane == L) zs = zl;
        }
      } else {  // internal levels: K1's own arithmetic
        double pT;
        if (dr.variant == VAR_B)
          pT = pass1<D, MASK, VAR_B>(dr, h, tab, P.ec, R, q, ck);
        else
          pT = pass1<D, MASK, VAR_C>(dr, h, tab, P.ec, R, q, ck);
        if (dr.n > 1) {
          const uint32_t c = (uint32_t)(M + di);
          const double u = P.randU ? P.randU[s * P.perU + c - 1] : philox_uniform(P.seed, (uint64_t)s, c);
          if (pT * scale < 1e-99) {
            const double w = dr.wts[dr.n - 1];
            double tot = 0.0;
            for (int z = 0; z < dr.n; ++z) tot += w;
            const double qv = w / tot;
            double cdf = 0.0;
            zs = dr.n - 1;
            bool found = false;
            for (int z = 0; z < dr.n - 1; ++z) {
              cdf += qv;
              if (!found && u <= cdf) {
                zs = z;
                found = true;
              }
            }
          } else {
            const double target = u * pT;
            int lo = 0, hi = dr.nchunks;
            while (lo < hi) {
              const int mid = (lo + hi) >> 1;
              if (target <= ck[mid]) hi = mid; else lo = mid + 1;
            }
            if (lo >= dr.nchunks) {
              zs = dr.n - 1;
            } else if (dr.G == 1) {
              zs = lo;
            } else {
              const double S0 = lo > 0 ? ck[lo - 1] : 0.0;
              if (dr.variant == VAR_B)
                zs = pass2<D, MASK, VAR_B>(dr, h, tab, P.ec, lo, S0, target);
              else
                zs = pass2<D, MASK, VAR_C>(dr, h, tab, P.ec, lo, S0, target);
            }
          }
        }
      }
      selpos[j] = zs;
      if (P.level_labels && dr.kind == 1 && live)
        P.level_labels[((s - P.s0) * M + j) * P.L + (dr.level - 1)] = dr.levperm[zs];

      {  // updateGlbParticlesVariance!(j)
        const double *rs = dr.rec_state + (size_t)zs * dr.state_stride;
#pragma unroll
        for (int k = 0; k < D; ++k) {
          const double var = dr.state_has_bw ? rs[D + k] : P.hvar[j][k];
          const double l = 1.0 / var;
          lam[j * D + k] = l;
          lmu[j * D + k] = rs[k] * l;
        }
      }
    }

    if (live) {  // labels (:612-616) and the final samplePoint! (:625)
      const int64_t o = s - P.s0;
      for (int j = 0; j < M; ++j) P.indices[o * M + j] = P.labels[j][selpos[j]];
#pragma unroll
      for (int k = 0; k < D; ++k) {
        double Lm = 0.0, Hm = 0.0;
        for (int i = 0; i < M; ++i) {
          Lm += lam[i * D + k];
          Hm += lmu[i * D + k];
        }
        double v = 0.0;
        const double cov = 1.0 / Lm;
        v = cov * Hm;
        if (P.add_entropy) {
          const uint32_t slot = (uint32_t)(P.L * D + k);
          const double g = P.randN ? P.randN[s * P.perN + slot] : philox_normal(P.seed, (uint64_t)s, slot);
          v = v + sqrt(cov) * g;
        }
        P.points[o * D + k] = v;
      }
    }
    batch = batch_next;
  }
  if (redone) atomicAdd(X.redone, (unsigned long long)redone);
  if (wredone) atomicAdd(X.warp_redone, (unsigned long long)wredone);
}

template <int D>
cudaError_t launch_gibbs_exact_d(const GibbsParams &P, const XParams &X, int grid, size_t smem, cudaStream_t st) {
  auto launch = [&](auto kern) -> cudaError_t {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
    if (e != cudaSuccess) return e;
    kern<<<grid, GB_THREADS, smem, st>>>(P, X);
    return cudaGetLastError();
  };
  if (P.M <= 4) return launch(gibbs_exact_kernel<D, 4>);
  if (P.M <= 8) return launch(gibbs_exact_kernel<D, 8>);
  return launch(gibbs_exact_kernel<D, KDEB200_MAX_DENS>);
}

// resident CTAs per SM of K1x at this d and M (the host sizes the grid and the redo scratch with it)
template <int D>
cudaError_t occupancy_gibbs_exact_d(int M, size_t smem, int *per_sm) {
  if (M <= 4) return cudaOccupancyMaxActiveBlocksPerMultiprocessor(per_sm, gibbs_exact_kernel<D, 4>, GB_THREADS, smem);
  if (M <= 8) return cudaOccupancyMaxActiveBlocksPerMultiprocessor(per_sm, gibbs_exact_kernel<D, 8>, GB_THREADS, smem);
  return cudaOccupancyMaxActiveBlocksPerMultiprocessor(per_sm, gibbs_exact_kernel<D, KDEB200_MAX_DENS>, GB_THREADS, smem);
}

}  // namespace kdeb200
