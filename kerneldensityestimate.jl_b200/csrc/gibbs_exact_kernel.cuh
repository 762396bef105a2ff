// gibbs_exact_kernel.cuh -- K1x (device code and launch template; gibbs_exact.cu holds the host side,
// gibbs_exact_d<N>.cu one explicit instantiation per d): the FP64 Gibbs sampler with every label DECIDED from certified
// FP32 prefix sums.
//
// Same schedule, chain state, RNG addressing and outputs as gibbs_kernel (K1), bit for bit.  K1 picks on every level
// the first z with target = fl(u * pT) <= S_z, S_z its sequential FP64 prefix sums (else n - 1).  On every draw -- leaf
// levels (variant A), the sampleIndices! draws (variant B) and the sampleIndex draws (variant C) of internal levels --
// K1x instead evaluates the nodes in packed FP32 (gibbs_f32_kernel.cuh's pair records and arithmetic) and carries next
// to every FP32 prefix sum S'_z a bound E_z on |S'_z - S_z / W| (W: the level's largest weight; DESIGN.md "K1x" derives
// it).  A lane's label is taken only when the intervals prove it:  hi(S_{z-1}) < lo(target)  and  hi(target) <= lo(S_z).
// A lane that cannot prove its label is redone by its warp with K1's FP64 node values, reading K1's exp table from
// global memory: first summed in parallel and certified again with an FP64-sized bound (xa_tier2), and only what that
// cannot prove summed by one lane in node order (xa_redo, K1w's scheme: K1's label by construction).
#pragma once
#include <type_traits>

#include "gibbs_f32_kernel.cuh"

namespace kdeb200 {

constexpr int GX_SCR = 256;   // nodes per block of the cooperative FP64 redo (its per-warp global scratch: GX_SCR doubles
                              // of terms, then one running sum per block)
// resident CTAs per SM the register budget is cut for: 4 (128 registers), the fastest of 4 / 5 / 6 / 8 at d = 3 now that
// no exp table limits the shared memory (DESIGN.md "K1x" has the sweep)
#ifndef GX_MINBLOCKS
#define GX_MINBLOCKS 4
#endif

// per-draw extras of K1x (certified draws only; zero elsewhere)
struct alignas(16) XDraw {
  const float *rec32;                 // FP32 pair records, coordinates relative to the tile centre
  const double *ctr;                  // tile centres, KDEB200_MAX_DIM doubles per tile of this draw
  double rad[KDEB200_MAX_DIM];        // max over the level of |m - centre| per dimension (FP64, rounded up)
  double bmin[KDEB200_MAX_DIM];       // variants B, C: the level's smallest node variance b_k per dimension
  double lw2max;                      // log2 of the level's largest weight (records hold lw2max - log2 w >= 0)
  int G, nchunks;                     // K1x's own checkpoint chunks (nodes, power of two)
  int fp32;                           // 0: the level is outside the FP32 range guard, every lane goes to xa_tier2
  int pad;
};

struct XParams {
  const XDraw *xd;
  double *scratch;                    // scr_stride doubles per warp of the grid
  unsigned long long *redone;         // leaf lane-draws redone in FP64 (live chains only)
  unsigned long long *warp_redone;    // leaf warp-draws with at least one redone lane
  unsigned long long *redone_int;     // the same two for the sampleIndex draws of internal levels (variant C)
  unsigned long long *warp_redone_int;
  unsigned long long *redone_b;       // the same two for the sampleIndices! draws (variant B)
  unsigned long long *warp_redone_b;
  unsigned long long *tier3;          // lane-draws (live chains) and warp-draws of every class that the warp-parallel
  unsigned long long *warp_tier3;     // FP64 sum (xa_tier2) could not decide and the serial sweep (xa_redo) did
  double ex2_err;                     // relative error bound of ex2.approx.ftz.f32 on [-126, 0]
  double rsq_err;                     // relative error bound of rsqrt.approx.ftz.f32 on normal floats
  double inflate;                     // test hook: multiplies the FP32 bound and xa_tier2's delta (1 in production)
  int scr_stride;                     // GX_SCR + the largest number of redo blocks of a level
};

// The bound of one certified draw: |p32 - p64 / W| <= p32 (A + B acc32) per node, plus aabs; prefix sums add the
// summation terms.  DESIGN.md "K1x" derives every constant.
struct XBound {
  double A, B, aabs, eta;
  bool ok;
};

// The per-chain FP32 constants of a certified draw, from K1's FP64 conditional (Calmost = cadd, leaf variances hvar):
//   ks: kernel-width scale per dimension (A: s_k = sqrt(0.5 log2e / c_k), c_k = hvar_k + Calmost_k; B: the same for the
//       level's narrowest b_min,k; C: for the level's narrowest c_k = b_min,k + Calmost_k), which measures the tile
//       radii of the bound;
//   sv: what the tile hoist clamps with (A: s_k; B, C: |mu - centre| <= 1e12 kernel widths);
//   g.a, g.c: A: s_k; B: 1; C: 1 and Calmost_k, so that gf_pre forms c_k = b_k + Calmost_k and
//       d_k = m'_k - (mu_k - centre_k);
//   rsmax: C: the largest normaliser prod_k c_k^-1/2 of the level (1 for A and B).
// Returns false when a variant-C chain's c_k could leave [2^-30, 2^30] (FP32 products of three of them stay normal), or
// a variant-B level's b_min,k lies below 2^-30 (the scale ks would be clamped, and the radii of the bound with it).
template <int D, int VAR>
__device__ __forceinline__ bool x_chain(const XDraw &xd, const double (&cadd)[D], const double *__restrict__ hvar,
                                        float (&ks)[D], float (&sv)[D], Hoist32<D> &g, double &rsmax) {
  bool ok = true;
  rsmax = 1.0;
#pragma unroll
  for (int k = 0; k < D; ++k) {
    if (VAR == VAR_A) {
      const float s = (float)sqrt(GF_HL2E / (hvar[k] + cadd[k]));  // c_k as K1 forms it
      ks[k] = sv[k] = s;
      g.a[k] = gf_pack(s, s);
    } else {
      const double cm = (VAR == VAR_B) ? xd.bmin[k] : xd.bmin[k] + cadd[k];  // <= every node's b_k / c_k
      // below 2^-30 the clamp in ks would shrink the radii of the bound: such a draw is not decided (both variants)
      ok = ok && cm >= 0x1.0p-30;
      if (VAR == VAR_C) ok = ok && cadd[k] <= 0x1.0p29;  // the host keeps b_k <= 2^29
      ks[k] = (float)sqrt(GF_HL2E / fmax(cm, 0x1.0p-30));
      sv[k] = (float)(1e12 / (double)ks[k]);
      rsmax *= cm;
      g.a[k] = gf_pack(1.f, 1.f);
      if (VAR == VAR_C) {
        const float cf = (float)cadd[k];
        g.c[k] = gf_pack(cf, cf);
      }
    }
  }
  rsmax = (VAR == VAR_C) ? 1.0 / sqrt(fmax(rsmax, 1e-300)) : 1.0;
  return ok;
}

template <int D, int VAR>
__device__ __forceinline__ XBound xa_bound(const XDraw &xd, const float (&ks)[D], double rsmax, int n, double ex2_err,
                                           double rsq_err, double inflate) {
  const double u = 0x1.0p-24 * (1.0 + 0x1.0p-20);
  double Rmax = 0.0, Rsum = 0.0, R2 = 0.0;
#pragma unroll
  for (int k = 0; k < D; ++k) {
    const double R = xd.rad[k] * (double)ks[k] * (1.0 + 3.0 * u);
    Rmax = fmax(Rmax, R);
    Rsum += R;
    R2 += R * R;
  }
  // variant C: d_k is one FFMA (4.02u on t^2 instead of A's 6.02u), c_k = b_k + Calmost_k 2.01u, the reciprocals from
  // rs^2 and two products 2 eps_rsq + 5u, D + 3 roundings of the non-negative sum.  Variant B: d_k as C (4.02u), the
  // record's 0.5 log2e / b_k 1.01u, the FMUL of d^2 u, D FFMA and lw' (D + 1)u: A's (D + 7.03)u
  constexpr int ng = (D + 3) / 4;  // rsqrt groups of gf_pre
  const double a1 = (VAR != VAR_C ? (D + 7.2) * u : (D + 14.2) * u + 2.02 * rsq_err) + 2.05 * u * Rmax;
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
  // variant C: the normaliser rs32 = fl(rsqrt(fl(prod c32))) against prod c^-1/2, and the product ex2 * rs32; K1's
  // own FP64 rsqrt, products and reciprocals as a further relative 1e-14
  const double norm = (VAR != VAR_C) ? 0.0 : 1.01 * (ng * rsq_err + (1.51 * D + 2.0 * ng) * u) + 1e-14;
  b.A = inflate * (1.003 * (ln2 * (a0 + 1.001 * a1 * a0) + 1.01 * ex2_err + norm) + 2.0 * gf_unr(D, VAR) * 1.01 * u +
                   (double)n * 0x1.0p-52 + 1e-15 * (6.0 + lwm));
  // ex2.approx.ftz flushes 2^-acc below 2^-126 to zero (variant C: times the normaliser, and the FP32 product may be
  // subnormal); K1 clamps exponents below -700 (kde_exp_flush)
  b.aabs = (VAR != VAR_C) ? 0x1.0p-125 + exp(-699.0 - xd.lw2max * ln2)
                          : 1.01 * (0x1.0p-125 * (1.0 + rsmax) + exp(-699.0 - xd.lw2max * ln2) * rsmax);
  b.eta = (double)n * 1.2e-16 + 1e-15;
  return b;
}

__device__ __forceinline__ double xa_err(const XBound &b, double S, double Q, int cnt) {
  return 1.01 * (b.A * S + b.B * Q) + (double)cnt * b.aabs;
}

// per tile: A: b_k = (mu_k - centre_k) s_k in FP64, clamped so that FP32 never sees an infinity; C: mu_k - centre_k,
// clamped to 1e12 kernel widths (sv)
template <int D, int VAR>
__device__ __forceinline__ void xa_tile_hoist(const double *__restrict__ ctr, const double (&mu)[D], const float (&sv)[D],
                                              Hoist32<D> &g) {
#pragma unroll
  for (int k = 0; k < D; ++k) {
    const double bk = (VAR == VAR_A) ? fmin(fmax((mu[k] - ctr[k]) * (double)sv[k], -1e12), 1e12)
                                     : fmin(fmax(mu[k] - ctr[k], -(double)sv[k]), (double)sv[k]);
    const float fb = (float)(-bk);
    g.b[k] = gf_pack(fb, fb);
  }
}

// one record pair -> the two FP32 terms and their exponents
template <int D, int VAR, bool NC>
__device__ __forceinline__ void xa_pair(const float *__restrict__ r, const Hoist32<D> &g, float &pa, float &pb, float &al,
                                        float &ah) {
  f32x2 acc, sc;
  gf_pre<D, VAR, NC>(r, g, acc, sc);
  gf_unpack(acc, al, ah);
  gf_fin<VAR>(acc, sc, pa, pb);
}

// pass 1 over the FP32 tiles of a certified draw: trip sums of 2 UNR terms in FP32 folded into an FP64 running sum,
// Q = sum p32 acc32 (the exponent-proportional part of the bound), both checkpointed every G nodes
template <int D, int VAR>
__device__ __forceinline__ double xa_pass1(const Draw &dr, const XDraw &xd, const double (&mu)[D], const float (&sv)[D],
                                           Hoist32<D> &g, Ring &R, int64_t &q, double *__restrict__ ck,
                                           float *__restrict__ ckq, double &Qout) {
  constexpr int UNR = gf_unr(D, VAR);
  constexpr int stride = gf_stride(D, VAR);
  const int npt = (dr.n + 1) >> 1;
  const int Gp = xd.G >> 1;
  const int tp = dr.tnodes >> 1;
  double S = 0.0, Q = 0.0;
  float qf = 0.f;
  int c = 0, done = 0, left = Gp;
  for (int t = 0; t < dr.ntiles; ++t, ++q) {
    xa_tile_hoist<D, VAR>(xd.ctr + (size_t)t * KDEB200_MAX_DIM, mu, sv, g);
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
        gf_trip_pre<D, VAR, UNR>(r + (size_t)i * stride, g, acc, sc);
        float s = 0.f;
#pragma unroll
        for (int uu = 0; uu < UNR; ++uu) {
          float al, ah, pa, pb;
          gf_unpack(acc[uu], al, ah);
          gf_fin<VAR>(acc[uu], sc[uu], pa, pb);
          s = __fadd_rn(s, pa);
          s = __fadd_rn(s, pb);
          qf = __fmaf_rn(pa, al, qf);
          qf = __fmaf_rn(pb, ah, qf);
        }
        S = __dadd_rn(S, (double)s);
      }
      for (; i < run; ++i) {
        float al, ah, pa, pb;
        xa_pair<D, VAR, false>(r + (size_t)i * stride, g, pa, pb, al, ah);
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
template <int D, int VAR>
__device__ __forceinline__ int xa_decide(const Draw &dr, const XDraw &xd, const XBound &bd, const double (&mu)[D],
                                         const float (&sv)[D], Hoist32<D> &g, const double *__restrict__ ck,
                                         const float *__restrict__ ckq, double tc, double tLo, double tHi) {
  constexpr int stride = gf_stride(D, VAR);
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
  int cur = -1;
  for (int z = z0; z < z1; z += 2) {
    const int t = z / dr.tnodes;
    if (t != cur) {
      xa_tile_hoist<D, VAR>(xd.ctr + (size_t)t * KDEB200_MAX_DIM, mu, sv, g);
      cur = t;
    }
    float al, ah, pa, pb;
    xa_pair<D, VAR, true>(xd.rec32 + (size_t)(z >> 1) * stride, g, pa, pb, al, ah);
    const float pp[2] = {pa, pb};
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

// K1's label when its pT * scale < 1e-99 rule fires (:311-315: all p[z] = weight(last node)); rare, lane 0 computes it
__device__ __forceinline__ int x_flat(const Draw &dr, double u) {
  const int n = dr.n;
  int zs = n - 1;
  if ((threadIdx.x & 31) == 0) {
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
  return __shfl_sync(0xffffffffu, zs, 0);
}

// Tier 2 of an undecided draw: K1's FP64 node values, summed by the whole warp in parallel, with a certificate.  One
// block of GX_SCR nodes: lane l evaluates nodes base + GX_RUN l .. + GX_RUN - 1 with K1's eval_node and adds them in
// order (p[i]: its run's partial sums); a warp scan of the run totals gives each lane the sum of the runs before it
// (excl) and the block total (tot).  Every term reaches p[i] through at most GX_RUN roundings, excl and tot through at
// most GX_RUN + 5.
constexpr int GX_RUN = GX_SCR / 32;
template <int D, int VAR>
__device__ __forceinline__ void x2_block(const Draw &dr, const Hoist<D, false> &h, const double *__restrict__ tab,
                                         const ExpConsts &ec, int base, double (&p)[GX_RUN], double &excl, double &tot) {
  const unsigned FULL = 0xffffffffu;
  const int lane = threadIdx.x & 31;
  const int z0 = base + lane * GX_RUN;
  double s = 0.0;
#pragma unroll
  for (int i = 0; i < GX_RUN; ++i) {
    if (z0 + i < dr.n) s = __dadd_rn(s, eval_node<D, false, VAR, true>(dr.rec + (size_t)(z0 + i) * dr.stride, h, tab, ec));
    p[i] = s;
  }
  double inc = s;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const double t = __shfl_up_sync(FULL, inc, o);
    if (lane >= o) inc = __dadd_rn(inc, t);
  }
  excl = __shfl_up_sync(FULL, inc, 1);
  if (lane == 0) excl = 0.0;
  tot = __shfl_sync(FULL, inc, 31);
}

// K1's label for one lane's undecided draw from the warp-parallel FP64 sums of x2_block, or -1 when they cannot prove
// it.  Block end-sums C_b = C_{b-1} + tot_b go to scr[GX_SCR + b]; node prefixes are C_{b-1} + (excl + p[i]).  Each
// computed sum S'_z is a sum of K1's non-negative terms through at most nb + GX_RUN + 7 roundings, K1's own S_z one
// through at most n, so S_z lies in S'_z [1 - delta, 1 + delta] with delta = 1.001 (n + nb + GX_RUN + 7) 2^-53
// (DESIGN.md "K1x" derives it; `inflate` scales it like the FP32 bound).  The label is taken as xa_decide takes it:
// the first node whose interval can reach the target, when its lower end provably reaches it (or it is node n - 1).
template <int D, int VAR>
__device__ __noinline__ int xa_tier2(const Draw &dr, const Hoist<D, false> &h, double scale, double u,
                                     const double *__restrict__ tab, const ExpConsts &ec, double *__restrict__ scr,
                                     double inflate) {
  const unsigned FULL = 0xffffffffu;
  const int lane = threadIdx.x & 31;
  const int n = dr.n;
  const int nb = (n + GX_SCR - 1) / GX_SCR;
  const double delta = inflate * 1.001 * (double)(n + nb + GX_RUN + 7) * 0x1.0p-53;
  const double fLo = __dadd_rd(1.0, -delta), fHi = __dadd_ru(1.0, delta);
  double p[GX_RUN], excl, tot, C = 0.0;
  for (int b = 0; b < nb; ++b) {
    x2_block<D, VAR>(dr, h, tab, ec, b * GX_SCR, p, excl, tot);
    C = __dadd_rn(C, tot);
    if (lane == 0) scr[GX_SCR + b] = C;
  }
  __syncwarp();
  // non-finite sums, a uniform outside [0, 1) (the target interval would not be ordered) and a 1e-99 rule that could
  // go either way are left to tier 3
  if (!isfinite(C) || !(u >= 0.0 && u < 1.0)) return -1;
  const double pLo = __dmul_rd(C, fLo), pHi = __dmul_ru(C, fHi);
  if (__dmul_ru(pHi, scale) < 1e-99) return x_flat(dr, u);  // K1's rule fires for every pT in the interval
  if (!(pLo > 0.0 && __dmul_rd(pLo, scale) >= 1e-99)) return -1;
  // K1's target fl(u pT) lies in [tLo, tHi]: fl is monotone, and rounds no lower than RD nor higher than RU
  const double tLo = __dmul_rd(u, pLo), tHi = __dmul_ru(u, pHi);
  unsigned bf = (unsigned)nb;  // first block whose end-sum interval reaches tLo; K1's sums before it all lie below
  for (int b = lane; b < nb; b += 32)
    if (tLo <= __dmul_ru(scr[GX_SCR + b], fHi)) {
      bf = (unsigned)b;
      break;
    }
  bf = __reduce_min_sync(FULL, bf);
  if (bf >= (unsigned)nb) return -1;
  const int base = (int)bf * GX_SCR;
  const double C0 = bf ? scr[GX_SCR + bf - 1] : 0.0;
  __syncwarp();  // scr is tier 3's to overwrite after this
  x2_block<D, VAR>(dr, h, tab, ec, base, p, excl, tot);
  // per lane the first of its nodes whose interval reaches tLo, key 2 z + (not certified); the warp takes the least z
  unsigned key = 0xffffffffu;
#pragma unroll
  for (int i = GX_RUN - 1; i >= 0; --i) {
    const int z = base + lane * GX_RUN + i;
    const double S = __dadd_rn(C0, __dadd_rn(excl, p[i]));
    if (z < n && tLo <= __dmul_ru(S, fHi)) key = 2u * (unsigned)z + ((tHi <= __dmul_rd(S, fLo) || z == n - 1) ? 0u : 1u);
  }
  key = __reduce_min_sync(FULL, key);
  return (key & 1u) ? -1 : (int)(key >> 1);
}

// Tier 3: K1's label for one lane's undecided draw, computed by the whole warp: lanes evaluate the nodes with K1's
// eval_node, lane 0 adds them in node order (the same additions as K1's pass 1 and pass 2), pT < 1e-99 rule included.
// The first sweep records the running sum at the end of every block of GX_SCR nodes (scr[GX_SCR + b]); the second sweep
// re-evaluates only the block whose end-sum first reaches the target, continuing from the exact sum before it.
template <int D, int VAR>
__device__ __noinline__ int xa_redo(const Draw &dr, const Hoist<D, false> &h, double scale, double u,
                                    const double *__restrict__ tab, const ExpConsts &ec, double *__restrict__ scr) {
  const unsigned FULL = 0xffffffffu;
  const int lane = threadIdx.x & 31;
  const int n = dr.n;
  const int nb = (n + GX_SCR - 1) / GX_SCR;
  double S = 0.0;
  for (int b = 0; b < nb; ++b) {
    const int base = b * GX_SCR;
    const int cnt = (n - base < GX_SCR) ? n - base : GX_SCR;
    for (int i = lane; i < cnt; i += 32) scr[i] = eval_node<D, false, VAR, true>(dr.rec + (size_t)(base + i) * dr.stride, h, tab, ec);
    __syncwarp();
    if (lane == 0) {
      for (int i = 0; i < cnt; ++i) S = __dadd_rn(S, scr[i]);
      scr[GX_SCR + b] = S;
    }
    __syncwarp();
  }
  const double pT = __shfl_sync(FULL, S, 0);
  int zs = n - 1;
  if (pT * scale < 1e-99) return x_flat(dr, u);  // :311-315: all p[z] = weight(last node)
  const double target = u * pT;
  unsigned bf = (unsigned)nb;  // first block whose end-sum reaches the target
  for (int b = lane; b < nb; b += 32)
    if (target <= scr[GX_SCR + b]) {
      bf = (unsigned)b;
      break;
    }
  bf = __reduce_min_sync(FULL, bf);
  if (bf >= (unsigned)nb) return zs;
  const int base = (int)bf * GX_SCR;
  const int cnt = (n - base < GX_SCR) ? n - base : GX_SCR;
  S = bf ? scr[GX_SCR + bf - 1] : 0.0;
  for (int i = lane; i < cnt; i += 32) scr[i] = eval_node<D, false, VAR, true>(dr.rec + (size_t)(base + i) * dr.stride, h, tab, ec);
  __syncwarp();
  int f = base + cnt - 1;
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
  return f;
}

// The FP64 tiers for the undecided lanes `ub` of a warp-draw, one lane at a time with the whole warp: tier 2
// (xa_tier2), and tier 3 (xa_redo) for what tier 2 cannot prove.  Returns this lane's label (z if it was decided in
// FP32).  Out of line with everything it needs, so that the hot loop's register allocation does not see it; tier 3 is
// rare at inflate 1, so its counters are global atomics here.
template <int D, int VAR>
__device__ __noinline__ int xa_undecided(const Draw &dr, unsigned ub, const double (&mu)[D], const double (&cadd)[D],
                                         const double *__restrict__ hvar, double scale, double u, bool live, int z,
                                         const double *__restrict__ tab, const ExpConsts &ec, double *__restrict__ scr,
                                         const XParams &X) {
  const unsigned FULL = 0xffffffffu;
  const int lane = threadIdx.x & 31;
  bool t3 = false;  // this warp-draw reached tier 3
  while (ub) {
    const int L = __ffs(ub) - 1;
    ub &= ub - 1;
    Hoist<D, false> hl;
#pragma unroll
    for (int k = 0; k < D; ++k) {
      hl.mu[k] = __shfl_sync(FULL, mu[k], L);
      hl.cadd[k] = __shfl_sync(FULL, cadd[k], L);
      hl.ich[k] = (VAR == VAR_A) ? sqrt(0.5 / (hvar[k] + hl.cadd[k])) : 0.0;  // K1's expression
      hl.act[k] = true;
    }
    const double sL = __shfl_sync(FULL, scale, L), uL = __shfl_sync(FULL, u, L);
    int zl = xa_tier2<D, VAR>(dr, hl, sL, uL, tab, ec, scr, X.inflate);
    if (zl < 0) {
      zl = xa_redo<D, VAR>(dr, hl, sL, uL, tab, ec, scr);
      if (__shfl_sync(FULL, (int)live, L) && lane == 0) atomicAdd(X.tier3, 1ull);
      t3 = true;
    }
    if (lane == L) z = zl;
  }
  if (t3 && lane == 0) atomicAdd(X.warp_tier3, 1ull);
  return z;
}

// K1's conditional of a draw, from the chain state and with K1's expressions (so its FP64 values are K1's): sampleIndices!
// (kind 0) evaluates against the level's point X, sampleIndex (kind 1) against the product of the other densities'
// selected kernels.  The certified draw calls it again where it needs Calmost after pass 1, instead of keeping it live.
template <int D, int MD>
__device__ __forceinline__ void x_cond(int kind, int j, int M, const double (&lam)[MD * D], const double (&lmu)[MD * D],
                                       const double (&X)[D], double (&mu)[D], double (&cadd)[D]) {
#pragma unroll
  for (int k = 0; k < D; ++k) {
    if (kind == 0) {
      mu[k] = X[k];
      cadd[k] = 0.0;
      continue;
    }
    double Lm = 0.0, Hm = 0.0;
    for (int i = 0; i < M; ++i) {
      if (i == j) continue;
      Lm += lam[i * D + k];
      Hm += lmu[i * D + k];
    }
    const double cov = 1.0 / Lm;  // M > 1 on this route
    cadd[k] = cov;
    mu[k] = cov * Hm;
  }
}

template <int D, int MD>
__global__ void __launch_bounds__(GB_THREADS, GX_MINBLOCKS) gibbs_exact_kernel(const __grid_constant__ GibbsParams P,
                                                                                   const __grid_constant__ XParams X) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  double *tiles = reinterpret_cast<double *>(smem_raw);
  __shared__ __align__(8) uint64_t bars[GB_STAGES];
  const int tid = threadIdx.x, lane = tid & 31;
  const int M = P.M;
  const unsigned FULL = 0xffffffffu;
  double *scr = X.scratch + ((size_t)blockIdx.x * (GB_THREADS / 32) + (tid >> 5)) * X.scr_stride;

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
  unsigned redone[3] = {0, 0, 0}, wredone[3] = {0, 0, 0};  // per variant

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

      // a certified draw: FP32 pass 1, the bound, the FP32 decision, the FP64 tiers for the lanes it leaves undecided
      auto certified = [&](auto var) -> int {
        constexpr int VAR = decltype(var)::value;
        const XDraw xd = X.xd[di];
        Hoist32<D> g;
        float ks[D], sv[D];
        double rsmax, mu[D];
        bool rok;
        {
          double cadd[D];
          x_cond<D, MD>(dr.kind, j, M, lam, lmu, X_, mu, cadd);
          rok = x_chain<D, VAR>(xd, cadd, P.hvar[j], ks, sv, g, rsmax);
        }
        double Qt;
        const double pT = xa_pass1<D, VAR>(dr, xd, mu, sv, g, R, q, ck, ckq, Qt);
        int z = 0;
        if (dr.n > 1) {
          const uint32_t c = (uint32_t)(M + di);
          const double u = P.randU ? P.randU[s * P.perU + c - 1] : philox_uniform(P.seed, (uint64_t)s, c);
          XBound bd = xa_bound<D, VAR>(xd, ks, rsmax, dr.n, X.ex2_err, X.rsq_err, X.inflate);
          bd.ok = bd.ok && rok;
          double scale = 1.0;  // K1's normaliser of a leaf draw; internal draws have none (K1's scale = 1)
          if (VAR == VAR_A) {
            double mu2[D], cadd[D], prod = 1.0;
            x_cond<D, MD>(dr.kind, j, M, lam, lmu, X_, mu2, cadd);
#pragma unroll
            for (int k = 0; k < D; ++k) prod *= P.hvar[j][k] + cadd[k];
            scale = kde_rsqrt(prod);
          }
          const double E = xa_err(bd, pT, Qt, dr.n);
          const double pLo = (pT - E) * (1.0 - bd.eta), pHi = (pT + E) * (1.0 + bd.eta);
          // K1's pT * scale < 1e-99 rule must provably not fire; u in [0, 1) keeps the target interval ordered
          bool und = !(bd.ok && u >= 0.0 && u < 1.0 && pLo > 0.0 && pLo * exp2(xd.lw2max) * scale >= 1.000001e-99);
          if (!und) {
            const double tLo = u * pLo * (1.0 - 0x1.0p-50), tHi = u * pHi * (1.0 + 0x1.0p-50);
            z = xa_decide<D, VAR>(dr, xd, bd, mu, sv, g, ck, ckq, u * pT, tLo, tHi);
            und = z < 0;
          }
          unsigned ub = __ballot_sync(FULL, und);
          if (ub) {
            if (live && und) ++redone[VAR];
            if (lane == 0) ++wredone[VAR];
            double cadd[D];
            x_cond<D, MD>(dr.kind, j, M, lam, lmu, X_, mu, cadd);
            z = xa_undecided<D, VAR>(dr, ub, mu, cadd, P.hvar[j], scale, u, live, z, P.exptab, P.ec, scr, X);
          }
        }
        return z;
      };
      int zs;
      if (dr.variant == VAR_A)
        zs = certified(std::integral_constant<int, VAR_A>());
      else if (dr.variant == VAR_B)
        zs = certified(std::integral_constant<int, VAR_B>());
      else
        zs = certified(std::integral_constant<int, VAR_C>());
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
  unsigned long long *const lanes_out[3] = {X.redone, X.redone_b, X.redone_int};
  unsigned long long *const warps_out[3] = {X.warp_redone, X.warp_redone_b, X.warp_redone_int};
#pragma unroll
  for (int v = 0; v < 3; ++v) {
    if (redone[v]) atomicAdd(lanes_out[v], (unsigned long long)redone[v]);
    if (wredone[v]) atomicAdd(warps_out[v], (unsigned long long)wredone[v]);
  }
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
