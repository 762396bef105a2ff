// tree.cuh -- device-resident BallTreeDensity: level-ordered SoA/AoS records (K3).
#pragma once
#include <cstdint>
#include <memory>
#include <vector>

#include "common.cuh"

namespace kdeb200 {

// One BFS level of a tree (the reference's levelList after l levelDown! steps,
// src/MSGibbs01.jl:500-523).  Offsets are in doubles from kdeb200_tree_s::d_buf.
struct Level {
  int64_t n = 0;      // nodes on this level
  int cls = 1;        // 0: every node is a leaf (uniform bandwidth => hoisted arithmetic), 1: general
  int64_t offW = 0;   // raw weights, n doubles                         (fallback path only)
  int64_t offA = -1;  // cls 0: records [m_0..m_{d-1}, ln w]            stride SA
  int64_t offB = -1;  // cls 1: records [m_k.., -0.5/b_k.., ln w - 0.5 sum ln b_k]   stride SC
  int64_t offC = -1;  // cls 1: records [m_k.., b_k.., ln w]            stride SC
  int64_t offP = 0;   // permutation of the level's nodes (0 for internal nodes), in d_levperm
};

}  // namespace kdeb200

namespace kdeb200 {
struct TreeDraws;  // gibbs_batch.cu
}

struct kdeb200_tree_s {
  int d = 0;
  int64_t N = 0;
  bool gibbs_ready = false; // level records present (kdeb200_tree_create); false for kdeb200_tree_create_eval
  bool degenerate = false;  // some bandwidth <= 0 or non-finite value: fast arithmetic not valid
  double hvar[KDEB200_MAX_DIM] = {0};  // the uniform leaf variances (bandwidthMin/Max[1:d])
  double root_mean[KDEB200_MAX_DIM] = {0};  // mean of node 1 (centre of the FP32 coordinates)
  double root_var[KDEB200_MAX_DIM] = {0};   // bandwidth (variance) of node 1: data spread + leaf bandwidth (FP32 Gibbs map)
  double extent[KDEB200_MAX_DIM] = {0};     // max_i |x_i - root_mean| per dimension (FP32 accuracy guard)
  int SA = 0, SC = 0, SE = 0;          // record strides in doubles (even => 16-byte aligned records)
  std::vector<kdeb200::Level> levels;  // levels[0] = {root}; levels[l], l = 1..depth
  int depth = 0;                       // last distinct level (all leaves)
  char *d_base = nullptr;              // the single device allocation everything below points into
  double *d_buf = nullptr;             // all level records
  size_t buf_doubles = 0;
  int64_t *d_labels = nullptr;  // deepest level, level order: permutation + 1 (src/MSGibbs01.jl:615)
  int64_t *d_levperm = nullptr; // every level, level order: permutation (labelsChoosen, src/MSGibbs01.jl:111)
  double *d_leaf = nullptr;     // leaf order (N+1..2N): [x_0..x_{d-1}, w], stride SE -- evalDirect's order
  int64_t *d_perm = nullptr;    // leaf order: original 0-based index
  float *d_leaf32 = nullptr;    // lazily built FP32 shadow of d_leaf (centred, pre-scaled), eval_f32.cu
  double *d_tilebox = nullptr;  // lazily built bounding boxes + weight sums of the component tiles (eval_pruned.cu)
  double *d_tilebox32 = nullptr;  // ... and of the component-pair tiles of the FP32 kernel
  double wtotal = 0.0;          // sum_i |w_i| (error bound of the pruned evaluation)
  double *d_cw = nullptr;       // lazily built: normalised cumulative weights in ORIGINAL point order (sample, extras.cu)
  int64_t *d_leaf_of = nullptr; // ... and original index -> leaf position (same allocation as d_cw)
  size_t device_bytes = 0;
  int slot = 0;                 // context slot that owns the device memory (0 = primary)
  int device = 0;               // ... and its CUDA device
  std::vector<int64_t> h_perm;  // host copy of d_perm (scatter of sharded LOO rows)
  kdeb200_tree_s *replica[KDEB200_MAX_GPUS] = {nullptr};  // copies on the other GPUs of the in-process set (lazy)
  std::shared_ptr<kdeb200::TreeDraws> batch_draws[2];  // lazily built Gibbs draw templates, [b_records] (gibbs_batch.cu)
};

namespace kdeb200 {
// the tree's records on the GPU of context `slot` (the handle itself for slot 0; otherwise a lazily made peer copy)
int tree_on(kdeb200_tree_t t, int slot, kdeb200_tree_t *out);
}
