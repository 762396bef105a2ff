// gibbs_plan.cuh -- host only: the static schedule the thread-per-chain Gibbs kernels (K1, K1f, K1x) share, and the
// only place that decides its checkpoint chunks and tiles.  Every chain runs the same draws: levels, then passes
// (0: sampleIndices!, 1..T: sampleIndex), then densities.  Chunk and tile sizes follow the format of the records a
// draw's tiles stream, which each route chooses per level:
//   FP64 records (K1 everywhere, K1x on internal levels): G from 1, at least one double group of pass 1 (gb_dg);
//     tiles of the largest power of two of nodes with tn * 2 * stride * 8 <= GB_TILE_BYTES.
//   FP32 pair records (K1f everywhere, K1x on leaf levels): G from 2, at least 4 * gf_unr nodes; tiles of the largest
//     power of two of nodes whose pairs fit a ring stage.  The records live in the schedule's own area, one 32-byte
//     aligned block per (density, tree level, variant); tiles address it by offset until it is allocated.
#pragma once
#include <cstring>
#include <vector>

#include "gibbs_f32_kernel.cuh"

namespace kdeb200 {

struct PlanBlock {
  int j, level, variant, tnodes;
  size_t off;  // floats into the record area
};
struct PlanTile {
  const double *src;  // FP64 records, or null: FP32 pairs at `off` floats into the record area
  size_t off;
  uint32_t bytes;
};
struct Plan {
  std::vector<Draw> draws;
  std::vector<int> block;  // per draw: its FP32 record block, -1 for FP64 records
  std::vector<PlanBlock> blocks;
  std::vector<PlanTile> tiles;
  size_t nfloats = 0;  // size of the record area
};

inline int plan_block(Plan &S, int j, int li, int var, int64_t n, int stride, int tn) {
  for (size_t b = 0; b < S.blocks.size(); ++b)
    if (S.blocks[b].j == j && S.blocks[b].level == li && S.blocks[b].variant == var) return (int)b;
  S.blocks.push_back(PlanBlock{j, li, var, tn, S.nfloats});
  S.nfloats = (S.nfloats + (size_t)((n + 1) / 2) * stride + 7) & ~(size_t)7;  // pass 2 reads with 256-bit loads
  return (int)S.blocks.size() - 1;
}

// b_records: pass 0 of internal levels reads the B records (-0.5/b precomputed), which hold no b for the mask logic
inline void plan_schedule(const kdeb200_tree_t *trees, int M, int L, int T, bool b_records, bool f32_leaf,
                          bool f32_internal, Plan &S) {
  const int d = trees[0]->d;
  for (int l = 1; l <= L; ++l)
    for (int pass = 0; pass <= T; ++pass)
      for (int j = 0; j < M; ++j) {
        const kdeb200_tree_s *t = trees[j];
        const int li = l < t->depth ? l : t->depth;
        const Level &lv = t->levels[li];
        Draw dr;
        std::memset(&dr, 0, sizeof(dr));
        dr.j = (short)j;
        dr.kind = pass == 0 ? 0 : 1;
        dr.level = (short)l;
        dr.new_level = (pass == 0 && j == 0) ? 1 : 0;
        dr.n = (int)lv.n;
        dr.wts = t->d_buf + lv.offW;
        dr.levperm = t->d_levperm + lv.offP;
        if (lv.cls == 0) {
          dr.variant = VAR_A;
          dr.rec = t->d_buf + lv.offA;
          dr.stride = t->SA;
          dr.rec_state = dr.rec;
          dr.state_stride = t->SA;
          dr.state_has_bw = 0;
        } else {
          dr.variant = (pass == 0 && b_records) ? VAR_B : VAR_C;
          dr.rec = t->d_buf + (dr.variant == VAR_B ? lv.offB : lv.offC);
          dr.stride = t->SC;
          dr.rec_state = t->d_buf + lv.offC;
          dr.state_stride = t->SC;
          dr.state_has_bw = 1;
        }
        dr.tile0 = (int)S.tiles.size();
        int blk = -1;
        if (lv.cls == 0 ? f32_leaf : f32_internal) {
          const int stride = gf_stride(d, dr.variant);
          int G = 2;
          while ((int64_t)G * GB_MAXCK < lv.n) G *= 2;
          const int want = 4 * gf_unr(d, dr.variant);  // at least two trips per chunk (x 1/2 and x 2 measured: +-1 %)
          if (G < want && lv.n >= 2 * want) G = want;
          dr.G = G;
          int tn = 2;
          while ((size_t)tn * stride * sizeof(float) <= GB_TILE_BYTES) tn *= 2;
          dr.tnodes = tn;
          blk = plan_block(S, j, li, dr.variant, lv.n, stride, tn);
          for (int64_t a = 0; a < lv.n; a += tn) {
            const int64_t cnt = (lv.n - a < tn) ? (lv.n - a) : tn;
            S.tiles.push_back(PlanTile{nullptr, S.blocks[blk].off + (size_t)(a / 2) * stride,
                                       (uint32_t)(((cnt + 1) / 2) * stride * sizeof(float))});
          }
        } else {
          int G = 1;
          while ((int64_t)G * GB_MAXCK < lv.n) G *= 2;
          const int dg = gb_dg(d, dr.variant);
          if (G < dg && lv.n >= 2 * dg) G = dg;  // pass 1 checkpoints per whole double group
          dr.G = G;
          int tn = 1;
          while (tn * 2 * dr.stride * 8 <= GB_TILE_BYTES) tn *= 2;
          dr.tnodes = tn;
          for (int64_t a = 0; a < lv.n; a += tn) {
            const int64_t cnt = (lv.n - a < tn) ? (lv.n - a) : tn;
            S.tiles.push_back(PlanTile{dr.rec + a * dr.stride, 0, (uint32_t)(cnt * dr.stride * sizeof(double))});
          }
        }
        dr.nchunks = (int)((lv.n + dr.G - 1) / dr.G);
        dr.ntiles = (int)((lv.n + dr.tnodes - 1) / dr.tnodes);
        S.draws.push_back(dr);
        S.block.push_back(blk);
      }
}

}  // namespace kdeb200
