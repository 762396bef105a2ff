// gibbs_batch_kernel.cuh -- K1b: many independent Gibbs product problems in one launch (device code and launch
// template; gibbs_batch.cu holds the host side, gibbs_batch_d<N>.cu one explicit instantiation per d).
//
// Mapping (DESIGN.md "K1b"): K1's arithmetic, one CTA per 128-chain block of ONE problem.  The grid is not
// persistent: CTA b finds its problem p by binary search over the prefix of ceil(Np / 128) blocks per problem and runs
// samples [128 (b - first_p), ...) of p; idle lanes replay the last chain, as in K1.  Each CTA streams p's own tile
// list through K1's ring (no batch counter, no look-ahead across batches), with Draw, TileDesc, Hoist, eval_node,
// Ring / ring_fill, pass1 and pass2 taken unchanged from gibbs_kernel.cuh.  The per-chain expressions below are K1's
// verbatim (state init, samplePoint!, hoist, the 1e-99 rule, the chunk search, the final point), and so are the Philox addressing
// (problem seed, local sample index) and the injected-stream indexing.  Every problem's outputs are those of K1 run on
// that problem alone, bit for bit.
// The same kernel at MD = 32 / 64 is K1m (DESIGN.md "K1m", host side gibbs_many.cu, instantiations gibbs_many_d<N>.cu):
// a single call of more than KDEB200_MAX_DENS densities, run as a one-problem launch over the call's sample slice.
#pragma once
#include "gibbs_kernel.cuh"

namespace kdeb200 {

// One problem of a batch, in device memory: what gibbs_device puts into GibbsParams for a single K1 call.  MDC is the
// capacity of the per-density arrays: KDEB200_MAX_DENS for K1b, 32 or 64 for the single call of more than
// KDEB200_MAX_DENS densities (gibbs_many.cu), which GibbsParams cannot describe.
template <int MDC>
struct alignas(16) BatchProbT {
  const Draw *draws;
  const TileDesc *tiles;
  const double *randU, *randN;  // the problem's injected streams or null (Philox)
  double *points;               // d x Np
  int64_t *indices;             // M x Np
  int64_t Np, perU, perN;
  uint64_t seed;
  int ndraws, ntiles, M, L, add_entropy, pad_;
  const double *root_rec[MDC];
  const int64_t *labels[MDC];
  double hvar[MDC][KDEB200_MAX_DIM];
  unsigned char mask[MDC][KDEB200_MAX_DIM];
  unsigned char other[MDC][KDEB200_MAX_DIM];
};
using BatchProb = BatchProbT<KDEB200_MAX_DENS>;
static_assert(sizeof(BatchProb) % 16 == 0, "BatchProb is copied to shared memory in 16-byte words");
static_assert(sizeof(BatchProbT<KDEB200_MAX_DENS_LARGE>) % 16 == 0, "BatchProbT is copied in 16-byte words");

// One launch: the problems of one (d, masked) class (K1b), or the one problem of a many-density single call.
struct BatchParams {
  const void *probs;  // BatchProbT<max(MD, KDEB200_MAX_DENS)>[nprob]
  const int *block0;  // nprob + 1 entries: first CTA of each problem, then the grid size
  int nprob;
  const double *exptab;
  ExpConsts ec;
  // Read only by the capacities above KDEB200_MAX_DENS, which run one problem, the single call's slice of samples
  // [s0, Np) (Np is then the slice's end, s1), with outputs at s - s0 and the optional labelsChoosen record
  // [(s1 - s0)][M][L] of K1 (GibbsParams::level_labels).
  int64_t s0;
  int64_t *level_labels;
};

// MD = capacity of the per-chain state in densities, as in K1: 4, 8 or 16 for K1b; 32 or 64 for the single call of
// more than KDEB200_MAX_DENS densities (ONE below), whose descriptor is a BatchProbT<MD>.
template <int D, bool MASK, int MD>
__global__ void __launch_bounds__(GB_THREADS, GB_MINBLOCKS) gibbs_batch_kernel(const __grid_constant__ BatchParams B) {
  constexpr bool ONE = MD > KDEB200_MAX_DENS;
  using Prob = BatchProbT<ONE ? MD : KDEB200_MAX_DENS>;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  double *tiles = reinterpret_cast<double *>(smem_raw);
  __shared__ __align__(16) double tab[KDE_EXP_TAB];
  __shared__ __align__(8) uint64_t bars[GB_STAGES];
  __shared__ Prob P;
  const int tid = threadIdx.x;

  int lo = 0, hi = B.nprob - 1;  // the last problem whose first block is <= blockIdx.x (every problem has a block)
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (B.block0[mid] <= (int)blockIdx.x) lo = mid; else hi = mid - 1;
  }
  {
    const int4 *src = reinterpret_cast<const int4 *>(static_cast<const Prob *>(B.probs) + lo);
    int4 *dst = reinterpret_cast<int4 *>(&P);
    for (int i = tid; i < (int)(sizeof(Prob) / 16); i += GB_THREADS) dst[i] = src[i];
  }
  for (int i = tid; i < KDE_EXP_TAB; i += GB_THREADS) tab[i] = B.exptab[i];
  if (tid == 0) {
    for (int s = 0; s < GB_STAGES; ++s) mbar_init(&bars[s], 1);
    mbar_fence_init();
  }
  __syncthreads();
  const int M = P.M;

  Ring R;
  R.tiles = tiles;
  R.bars = bars;
  R.descs = P.tiles;
  R.ntiles = P.ntiles;
  R.known = P.ntiles;
  R.issued = 0;
  R.nxt = P.tiles[0];
  R.nxt_idx = 0;
  if (tid == 0) ring_fill(R, 0);
  int64_t q = 0;

  // chain state: lambda = 1/variance and lambda*mu of the currently selected node of each density
  double lam[MD * D];
  double lmu[MD * D];
  double ck[GB_MAXCK];
  int selpos[MD];

  int64_t s = (int64_t)((int)blockIdx.x - B.block0[lo]) * GB_THREADS + tid;
  if constexpr (ONE) s += B.s0;
  const bool live = s < P.Np;
  if (!live) s = P.Np - 1;  // idle lanes replay the last chain (keeps the CTA in lock-step)

  // levelInit!/initIndices!/calcIndices!: every density starts at the root
  for (int j = 0; j < M; ++j) {
    const double *rr = P.root_rec[j];
#pragma unroll
    for (int k = 0; k < D; ++k) {
      if (MASK && !P.mask[j][k]) {
        lam[j * D + k] = 0.0;
        lmu[j * D + k] = 0.0;
      } else {
        const double l = 1.0 / rr[D + k];
        lam[j * D + k] = l;
        lmu[j * D + k] = rr[k] * l;
      }
    }
    selpos[j] = 0;
  }

  double X[D];
  for (int di = 0; di < P.ndraws; ++di) {
    const Draw dr = P.draws[di];
    const int j = dr.j;

    if (dr.new_level) {  // samplePoint!(addEntropy = true) with normals g(level-1, k)
#pragma unroll
      for (int k = 0; k < D; ++k) {
        double Lm = 0.0, Hm = 0.0;
        bool any = !MASK;
        for (int i = 0; i < M; ++i) {
          if (MASK && P.mask[i][k]) any = true;
          Lm += lam[i * D + k];
          Hm += lmu[i * D + k];
        }
        const uint32_t slot = (uint32_t)((dr.level - 1) * D + k);
        const double g = P.randN ? P.randN[s * P.perN + slot] : philox_normal(P.seed, (uint64_t)s, slot);
        if (any) {
          const double cov = 1.0 / Lm;
          X[k] = cov * Hm + sqrt(cov) * g;
        } else {
          X[k] = 0.0;
        }
      }
    }

    Hoist<D, MASK> h;
    double scale = 1.0;  // normaliser common to the whole level (variant A), for the 1e-99 test
    if (dr.kind == 0) {
#pragma unroll
      for (int k = 0; k < D; ++k) {
        h.mu[k] = X[k];
        h.cadd[k] = 0.0;
        h.act[k] = MASK ? (P.mask[j][k] && P.other[j][k]) : true;
      }
    } else {  // leave-one-out product of the other densities' selected kernels
#pragma unroll
      for (int k = 0; k < D; ++k) {
        double Lm = 0.0, Hm = 0.0;
        for (int i = 0; i < M; ++i) {
          if (i == j) continue;
          Lm += lam[i * D + k];
          Hm += lmu[i * D + k];
        }
        const bool oth = MASK ? (P.other[j][k] != 0) : (M > 1);
        if (oth) {
          const double cov = 1.0 / Lm;
          h.cadd[k] = cov;
          h.mu[k] = cov * Hm;
        } else {
          h.cadd[k] = 0.0;
          h.mu[k] = 0.0;
        }
        h.act[k] = (MASK ? (P.mask[j][k] != 0) : true) && oth;
      }
    }
    if (dr.variant == VAR_A) {
      double prod = 1.0;
#pragma unroll
      for (int k = 0; k < D; ++k) {
        const double c = P.hvar[j][k] + h.cadd[k];
        h.ich[k] = sqrt(0.5 / c);
        if (!MASK || h.act[k]) prod *= c;
      }
      scale = kde_rsqrt(prod);
    }

    double pT;
    if (dr.variant == VAR_A)
      pT = pass1<D, MASK, VAR_A>(dr, h, tab, B.ec, R, q, ck);
    else if (dr.variant == VAR_B)
      pT = pass1<D, MASK, VAR_B>(dr, h, tab, B.ec, R, q, ck);
    else
      pT = pass1<D, MASK, VAR_C>(dr, h, tab, B.ec, R, q, ck);

    // selectLabelOnLevel: the c-th call of this chain reads randU[(s*perU + c) - 1]
    int zs = 0;
    if (dr.n > 1) {
      const uint32_t c = (uint32_t)(M + di);
      const double u = P.randU ? P.randU[s * P.perU + c - 1] : philox_uniform(P.seed, (uint64_t)s, c);
      if (pT * scale < 1e-99) {  // :311-315: all p[z] = weight(last node)
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
        int clo = 0, chi = dr.nchunks;  // first chunk whose end-prefix reaches the target
        while (clo < chi) {
          const int mid = (clo + chi) >> 1;
          if (target <= ck[mid]) chi = mid; else clo = mid + 1;
        }
        if (clo >= dr.nchunks) {
          zs = dr.n - 1;
        } else if (dr.G == 1) {
          zs = clo;
        } else {
          const double S0 = clo > 0 ? ck[clo - 1] : 0.0;
          if (dr.variant == VAR_A)
            zs = pass2<D, MASK, VAR_A>(dr, h, tab, B.ec, clo, S0, target);
          else if (dr.variant == VAR_B)
            zs = pass2<D, MASK, VAR_B>(dr, h, tab, B.ec, clo, S0, target);
          else
            zs = pass2<D, MASK, VAR_C>(dr, h, tab, B.ec, clo, S0, target);
        }
      }
    }
    selpos[j] = zs;
    if constexpr (ONE) {  // sampleIndex records permutation[ind[j]] per (sample, density, level), as in K1
      if (B.level_labels && dr.kind == 1 && live)
        B.level_labels[((s - B.s0) * M + j) * P.L + (dr.level - 1)] = dr.levperm[zs];
    }

    // updateGlbParticlesVariance!(j)
    {
      const double *rs = dr.rec_state + (size_t)zs * dr.state_stride;
#pragma unroll
      for (int k = 0; k < D; ++k) {
        if (MASK && !P.mask[j][k]) {
          lam[j * D + k] = 0.0;
          lmu[j * D + k] = 0.0;
        } else {
          const double var = dr.state_has_bw ? rs[D + k] : P.hvar[j][k];
          const double l = 1.0 / var;
          lam[j * D + k] = l;
          lmu[j * D + k] = rs[k] * l;
        }
      }
    }
  }

  // labels (:612-616) and the final samplePoint! (:625).  The descriptor's fields are taken into registers first: with
  // them in shared memory, nvcc cannot prove them unchanged across the stores below, and the point's expression then
  // contracts differently from K1's (where they are kernel parameters) in the last bit.
  const int L = P.L, add_entropy = P.add_entropy;
  const int64_t perN = P.perN;
  const uint64_t seed = P.seed;
  const double *randN = P.randN;
  double *points = P.points;
  int64_t *indices = P.indices;
  if (live) {
    int64_t o = s;
    if constexpr (ONE) o -= B.s0;
    for (int j = 0; j < M; ++j) indices[o * M + j] = P.labels[j][selpos[j]];
#pragma unroll
    for (int k = 0; k < D; ++k) {
      double Lm = 0.0, Hm = 0.0;
      bool any = !MASK;
      for (int i = 0; i < M; ++i) {
        if (MASK && P.mask[i][k]) any = true;
        Lm += lam[i * D + k];
        Hm += lmu[i * D + k];
      }
      double v = 0.0;
      if (any) {
        const double cov = 1.0 / Lm;
        v = cov * Hm;
        if (add_entropy) {
          const uint32_t slot = (uint32_t)(L * D + k);
          const double g = randN ? randN[s * perN + slot] : philox_normal(seed, (uint64_t)s, slot);
          v = v + sqrt(cov) * g;
        }
      }
      points[o * D + k] = v;
    }
  }
}

// one launch of `grid` CTAs for the problems of one (d, masked) class; MD from the class's largest M
template <int D>
cudaError_t launch_gibbs_batch_d(const BatchParams &B, bool masked, int maxM, int grid, cudaStream_t st) {
  const size_t smem = GB_STAGES * GB_TILE_BYTES;
  auto launch = [&](auto kern) -> cudaError_t {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
    if (e != cudaSuccess) return e;
    kern<<<grid, GB_THREADS, smem, st>>>(B);
    return cudaGetLastError();
  };
  if (masked) return launch(gibbs_batch_kernel<D, true, KDEB200_MAX_DENS>);
  if (maxM <= 4) return launch(gibbs_batch_kernel<D, false, 4>);
  if (maxM <= 8) return launch(gibbs_batch_kernel<D, false, 8>);
  return launch(gibbs_batch_kernel<D, false, KDEB200_MAX_DENS>);
}

// the single call of M > KDEB200_MAX_DENS densities (gibbs_many.cu): one problem, MD = 32 or 64 from M
template <int D>
cudaError_t launch_gibbs_many_d(const BatchParams &B, bool masked, int M, int grid, cudaStream_t st) {
  const size_t smem = GB_STAGES * GB_TILE_BYTES;
  auto launch = [&](auto kern) -> cudaError_t {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
    if (e != cudaSuccess) return e;
    kern<<<grid, GB_THREADS, smem, st>>>(B);
    return cudaGetLastError();
  };
  static_assert(KDEB200_MAX_DENS_LARGE == 64, "the instantiated capacities are 32 and 64");
  if (masked) return M <= 32 ? launch(gibbs_batch_kernel<D, true, 32>) : launch(gibbs_batch_kernel<D, true, 64>);
  return M <= 32 ? launch(gibbs_batch_kernel<D, false, 32>) : launch(gibbs_batch_kernel<D, false, 64>);
}

}  // namespace kdeb200
