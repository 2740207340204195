// Replay half of the hot path: float64 sum tree, sampling, gather, insert, priority write-back.
// Restates (on the device) dqn_zoo/replay.py:44-117 (UniformDistribution), :246-426 (SumTree),
// :429-651 (PrioritizedDistribution), :654-768 (PrioritizedTransitionReplay).  All float64
// arithmetic that feeds an index decision uses explicit round-to-nearest intrinsics so nvcc
// cannot contract a*b+c into an FMA: results are bit-identical to numpy's.
#include <map>
#include <vector>

#include "dz_internal.cuh"

namespace dz {

thread_local std::string g_last_error;
std::atomic<int64_t> g_launches{0};
std::vector<timeline_setter_t>& timeline_setters() { static std::vector<timeline_setter_t> v; return v; }
void timeline_register(timeline_setter_t fn) { timeline_setters().push_back(fn); }
int g_pdl = -1;
int g_carveout = -1;
bool g_profile = false;

namespace {
struct ProfileRec { const char* name; cudaEvent_t a, b; unsigned gx, gy, bx; };
std::vector<ProfileRec> g_profile_recs;
}  // namespace

void profile_geometry(unsigned gx, unsigned gy, unsigned bx) {
  if (!g_profile_recs.empty()) { g_profile_recs.back().gx = gx; g_profile_recs.back().gy = gy; g_profile_recs.back().bx = bx; }
}

void profile_mark(const char* name, void* stream, bool begin) {
  if (begin) {
    ProfileRec r{name, nullptr, nullptr, 0, 0, 0};
    cudaEventCreate(&r.a);
    cudaEventCreate(&r.b);
    cudaEventRecord(r.a, (cudaStream_t)stream);
    g_profile_recs.push_back(r);
  } else if (!g_profile_recs.empty()) {
    cudaEventRecord(g_profile_recs.back().b, (cudaStream_t)stream);
  }
}

// ------------------------------------------------------------------------------------------------
// Sum tree device routines
// ------------------------------------------------------------------------------------------------

__device__ __forceinline__ int tree_depth(int64_t first_leaf) { return 63 - __clzll(first_leaf); }

__device__ __forceinline__ bool finite_nonneg(double v) { return v >= 0.0 && v <= 1.7976931348623157e308; }

// Block-cooperative SumTree.set for n <= blockDim.x*ITEMS entries held in shared memory.
// s_idx[i] < 0 marks an entry to skip.  Leaves: last write wins (numpy fancy assignment,
// replay.py:283); then one pass per level, all ancestors recomputed as fl(left+right).
__device__ void block_tree_set(double* __restrict__ nodes, int64_t first_leaf, const int64_t* s_idx,
                               const double* s_val, int n) {
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    int64_t me = s_idx[i];
    if (me < 0) continue;
    bool last = true;
    for (int j = i + 1; j < n; ++j)
      if (s_idx[j] == me) { last = false; break; }
    if (last) nodes[first_leaf + me] = s_val[i];
  }
  __syncthreads();
  for (int shift = 1; (first_leaf >> shift) >= 1; ++shift) {  // parents of the leaves ... root
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
      int64_t me = s_idx[i];
      if (me < 0) continue;
      int64_t p = (first_leaf + me) >> shift;
      nodes[p] = __dadd_rn(nodes[2 * p], nodes[2 * p + 1]);
    }
    __syncthreads();
  }
}

constexpr int kSetChunk = 1024;

__global__ void __launch_bounds__(256) sumtree_set_kernel(double* nodes, int64_t first_leaf, int64_t size,
                                                          const int64_t* __restrict__ idx,
                                                          const double* __restrict__ vals, int n, int32_t* flags) {
  dz::pdl_enter();
  __shared__ int64_t s_idx[kSetChunk];
  __shared__ double s_val[kSetChunk];
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    int64_t k = idx[i];
    double v = vals[i];
    int bad = 0;
    if (!finite_nonneg(v)) bad |= DZ_FLAG_BAD_VALUE;
    if (k < 0 || k >= size) bad |= DZ_FLAG_BAD_INDEX;
    if (bad && flags) atomicOr(flags, bad);
    s_idx[i] = bad ? -1 : k;
    s_val[i] = v;
  }
  __syncthreads();
  block_tree_set(nodes, first_leaf, s_idx, s_val, n);
}

// update_priorities: `_power` in float32 (SURVEY §8(a) R3) then widen, then set.
__device__ __forceinline__ double exponentiate_f32(float p, double alpha) {
  if (p == 0.0f) return 0.0;  // 0**0 == 0 (replay.py:203-208)
  float r;
  if (alpha == 0.5) r = __fsqrt_rn(p);
  else if (alpha == 1.0) r = p;
  else r = (float)pow((double)p, (double)(float)alpha);  // canonical: round_f32(pow_f64(x,(double)(float)alpha))
  return (double)r;
}

__global__ void __launch_bounds__(256) update_priorities_kernel(double* nodes, int64_t first_leaf, int64_t size,
                                                                const int64_t* __restrict__ idx,
                                                                const float* __restrict__ pri, int n, double alpha,
                                                                int32_t* flags) {
  dz::pdl_enter();
  __shared__ int64_t s_idx[kSetChunk];
  __shared__ double s_val[kSetChunk];
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    int64_t k = idx[i];
    float p = pri[i];
    int bad = 0;
    if (!(p >= 0.0f && p <= 3.402823466e38f)) bad |= DZ_FLAG_BAD_VALUE;
    if (k < 0 || k >= size) bad |= DZ_FLAG_BAD_INDEX;
    if (bad && flags) atomicOr(flags, bad);
    s_idx[i] = bad ? -1 : k;
    s_val[i] = bad ? 0.0 : exponentiate_f32(p, alpha);
  }
  __syncthreads();
  block_tree_set(nodes, first_leaf, s_idx, s_val, n);
}

// Single-warp SumTree.set for n <= 32 float32 priorities (the learner's per-step write-back).  All 20
// sibling values of every path are prefetched with independent loads first; the bottom-up resum then
// runs in registers: lanes that share a parent find each other with __match_any_sync and take the
// sibling's NEW value from the other lane when the sibling is itself on an updated path, else the
// prefetched one.  Same fl(left+right) per node as the reference, ~3 dependent memory round trips
// instead of 2 per level.
__global__ void __launch_bounds__(32) update_priorities_warp_kernel(double* nodes, int64_t first_leaf, int64_t size,
                                                                    const int64_t* __restrict__ idx,
                                                                    const float* __restrict__ pri, int n, double alpha,
                                                                    int32_t* flags) {
  dz::pdl_enter();
  const unsigned full = 0xffffffffu;
  const int lane = threadIdx.x;
  int64_t k = -1;
  double val = 0.0;
  if (lane < n) {
    k = idx[lane];
    float p = pri[lane];
    int bad = 0;
    if (!(p >= 0.0f && p <= 3.402823466e38f)) bad |= DZ_FLAG_BAD_VALUE;
    if (k < 0 || k >= size) bad |= DZ_FLAG_BAD_INDEX;
    if (bad) { if (flags) atomicOr(flags, bad); k = -1; }
    else val = exponentiate_f32(p, alpha);
  }
  const bool active = k >= 0;
  const int depth = tree_depth(first_leaf);
  int64_t node = active ? first_leaf + k : (int64_t)(-2 - lane);   // inactive lanes get unique negative keys
  // prefetch the sibling of every node on this lane's path (values untouched by this update unless the
  // sibling is on another lane's path, in which case that lane's value is used instead)
  double sib[40];
#pragma unroll
  for (int l = 0; l < 40; ++l) sib[l] = 0.0;
  if (active) {
#pragma unroll
    for (int l = 0; l < 40; ++l)
      if (l < depth) sib[l] = nodes[(node >> l) ^ 1];
  }
  // duplicates: the highest lane (last in the batch) wins (numpy fancy assignment, replay.py:283)
  unsigned same = __match_any_sync(full, node);
  int winner = 31 - __clz((int)same);
  val = __shfl_sync(full, val, winner);
  if (active && lane == winner) nodes[node] = val;
#pragma unroll
  for (int l = 0; l < 40; ++l) {
    if (l >= depth) break;
    const int64_t parent = active ? (node >> 1) : node;
    const unsigned grp = __match_any_sync(full, parent);
    const unsigned is_left = __ballot_sync(full, active && ((node & 1) == 0));
    const unsigned lefts = grp & is_left, rights = grp & ~is_left;
    double lv = (node & 1) == 0 ? val : sib[l], rv = (node & 1) ? val : sib[l];
    const int lsrc = lefts ? __ffs((int)lefts) - 1 : lane, rsrc = rights ? __ffs((int)rights) - 1 : lane;
    double lo = __shfl_sync(full, val, lsrc), ro = __shfl_sync(full, val, rsrc);
    if (lefts) lv = lo;
    if (rights) rv = ro;
    const double sum = __dadd_rn(lv, rv);
    if (active && lane == __ffs((int)grp) - 1) nodes[parent] = sum;
    if (active) { node = parent; val = sum; }
  }
}

// Level-by-level rebuild (replay.py:394-404).  One launch per level keeps it simple and is only
// used by set_all / resize / set_state (never on the hot path).
__global__ void sumtree_zero_tail_kernel(double* nodes, int64_t first_leaf, int64_t n_valid) {
  dz::pdl_enter();
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x + n_valid;
  if (i < first_leaf) nodes[first_leaf + i] = 0.0;
  if (blockIdx.x == 0 && threadIdx.x == 0) nodes[0] = 0.0;
}
__global__ void sumtree_level_kernel(double* nodes, int64_t width) {
  dz::pdl_enter();
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i < width) {
    int64_t p = width + i;
    nodes[p] = __dadd_rn(nodes[2 * p], nodes[2 * p + 1]);
  }
}
// Top of the tree (<= 2048 leaves under it) in one block.
__global__ void __launch_bounds__(1024) sumtree_top_kernel(double* nodes, int64_t width_start) {
  dz::pdl_enter();
  for (int64_t width = width_start; width >= 1; width >>= 1) {
    for (int64_t i = threadIdx.x; i < width; i += blockDim.x) {
      int64_t p = width + i;
      nodes[p] = __dadd_rn(nodes[2 * p], nodes[2 * p + 1]);
    }
    __syncthreads();
  }
}

// Warp-cooperative descent (replay.py:406-426): the warp fetches up to five levels below the
// current node with two coalesced loads (2+4+8+16 children sums in lanes 0..29, the 32
// great^4-grandchildren in a second register), then walks them with shuffles.  A depth-20 tree
// costs 4 dependent memory round trips instead of 20.
__device__ int64_t warp_tree_descend(const double* __restrict__ nodes, int depth, double target) {
  const unsigned lane = threadIdx.x & 31u;
  int64_t node = 1;
  int level = 0;
  const int k_mine = 31 - __clz((int)lane + 2);        // sub-level served by this lane in register A
  const int r_mine = ((int)lane + 2) - (1 << k_mine);
  while (level < depth) {
    const int span = min(5, depth - level);
    double va = 0.0, vb = 0.0;
    if (k_mine <= 4 && k_mine <= span) va = nodes[(node << k_mine) + r_mine];
    if (span == 5) vb = nodes[(node << 5) + lane];
    int rel = 0;
    for (int k = 1; k <= span; ++k) {
      double left = (k <= 4) ? __shfl_sync(0xffffffffu, va, (1 << k) - 2 + 2 * rel)
                             : __shfl_sync(0xffffffffu, vb, 2 * rel);
      if (target < left) {
        rel = 2 * rel;
      } else {
        target = __dsub_rn(target, left);
        rel = 2 * rel + 1;
      }
    }
    node = (node << span) + rel;
    level += span;
  }
  return node;
}


__global__ void __launch_bounds__(256) sumtree_query_kernel(const double* __restrict__ nodes, int64_t first_leaf,
                                                            const double* __restrict__ targets, int64_t n,
                                                            int64_t* __restrict__ out, int32_t* flags) {
  dz::pdl_enter();
  int64_t q = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
  if (q >= n) return;
  double root = nodes[1];
  double t = targets[q];
  if (!(t >= 0.0 && t < root)) {  // replay.py:408-409
    if ((threadIdx.x & 31) == 0) {
      if (flags) atomicOr(flags, DZ_FLAG_BAD_TARGET);
      out[q] = -1;
    }
    return;
  }
  int64_t node = warp_tree_descend(nodes, tree_depth(first_leaf), t);
  if ((threadIdx.x & 31) == 0) out[q] = node - first_leaf;
}

__global__ void sumtree_get_kernel(const double* __restrict__ nodes, int64_t first_leaf, int64_t size,
                                   const int64_t* __restrict__ idx, int64_t n, double* __restrict__ out,
                                   int32_t* flags) {
  dz::pdl_enter();
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= n) return;
  int64_t k = idx[i];
  if (k < 0 || k >= size) {
    if (flags) atomicOr(flags, DZ_FLAG_BAD_INDEX);
    out[i] = 0.0;
    return;
  }
  out[i] = nodes[first_leaf + k];
}

// ------------------------------------------------------------------------------------------------
// Sampling (replay.py:547-583 + :706-717, and :76-82)
// ------------------------------------------------------------------------------------------------

__device__ __forceinline__ double is_weight_pow(double x, double beta) {
  // numpy's `**` with a scalar exponent takes exact shortcuts for 1, 0.5 and 0; mirror them.
  if (beta == 1.0) return x;
  if (beta == 0.5) return __dsqrt_rn(x);
  if (beta == 0.0) return 1.0;
  return pow(x, beta);
}

__device__ void emit_batch_rows(const dz_replay_view& v, const BatchExtras& ex, int b, int64_t slot, double weight) {
  if (v.frames.d_frames) {   // frame store: the stacks are assembled into fixed staging rows after the sampler
    const uint8_t* row = v.frames.d_batch_stage + (int64_t)b * v.obs_stride;
    if (ex.d_s_tm1_rows) ex.d_s_tm1_rows[b] = row;
    if (ex.d_s_t_rows) ex.d_s_t_rows[b] = row + (int64_t)v.frames.batch_capacity * v.obs_stride;
  } else {
    const uint8_t* row = v.d_obs + slot * 2 * v.obs_stride;
    if (ex.d_s_tm1_rows) ex.d_s_tm1_rows[b] = row;
    if (ex.d_s_t_rows) ex.d_s_t_rows[b] = row + v.obs_stride;
  }
  if (ex.d_a) ex.d_a[b] = v.d_action[slot];
  if (ex.d_r) ex.d_r[b] = (float)v.d_reward[slot];      // float64 -> float32 at the jit boundary
  if (ex.d_disc) ex.d_disc[b] = (float)v.d_discount[slot];
  if (ex.d_w) ex.d_w[b] = (float)weight;
}

__global__ void __launch_bounds__(1024) per_sample_kernel(dz_replay_view v, dz_sample_inputs in, dz_sample_outputs out,
                                                          int batch, BatchExtras ex) {
  dz::pdl_enter();
  extern __shared__ double s_w[];  // [batch] unnormalised weights
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = blockDim.x >> 5;
  const double* nodes = v.d_tree;
  const double root = nodes[1];
  const int64_t size = (int64_t)in.d_scalars[0];
  const double beta = in.d_scalars[1];
  const double usp = in.d_scalars[2];
  const bool normalize = in.d_scalars[3] != 0.0;
  const double one_over_n = __ddiv_rn(1.0, (double)size);
  const int depth = tree_depth(v.first_leaf);
  for (int q = warp; q < batch; q += nwarps) {
    int64_t pos = in.d_rand_pos[q];
    int64_t uni = v.d_live[pos];
    int64_t pri;
    if (root == 0.0) {  // replay.py:556-557 (the host must then skip the second RNG draw)
      pri = uni;
      if (lane == 0 && v.d_flags && ex.fused) atomicOr(v.d_flags, DZ_FLAG_ROOT_ZERO);
    } else {
      double target = __dmul_rn(in.d_u_tree[q], root);
      if (!(target >= 0.0 && target < root)) {
        if (lane == 0 && v.d_flags) atomicOr(v.d_flags, DZ_FLAG_BAD_TARGET);
        target = 0.0;
      }
      pri = warp_tree_descend(nodes, depth, target) - v.first_leaf;
    }
    int64_t idx = (in.d_u_mix[q] < usp) ? uni : pri;
    double leaf = nodes[v.first_leaf + idx];
    double frac = (root == 0.0) ? one_over_n : __ddiv_rn(leaf, root);
    double prob = __dadd_rn(__dmul_rn(__dsub_rn(1.0, usp), frac), __dmul_rn(usp, one_over_n));
    if (lane == 0) {
      int64_t id = v.d_id_at[idx];
      const int64_t slot = id % v.capacity;
      out.d_indices[q] = idx;
      out.d_ids[q] = id;
      out.d_slots[q] = slot;
      out.d_probs[q] = prob;
      // row pointers and scalars of the sampled transition do not depend on the batch-wide weight normalisation: their
      // (DRAM-latency) loads are issued here, under the pow() and the block reduction, instead of after them
      emit_batch_rows(v, ex, q, slot, 0.0);
      s_w[q] = is_weight_pow(__ddiv_rn(one_over_n, prob), beta);
    }
  }
  __syncthreads();
  // importance_sampling_weights (replay.py:238-243): optional division by the batch max.
  __shared__ double s_max[32];
  double m = 0.0;
  for (int q = threadIdx.x; q < batch; q += blockDim.x) m = fmax(m, s_w[q]);
  m = warp_max(m);
  if (lane == 0) s_max[warp] = m;
  __syncthreads();
  if (warp == 0) {
    m = (lane < nwarps) ? s_max[lane] : 0.0;
    m = warp_max(m);
    if (lane == 0) s_max[0] = m;
  }
  __syncthreads();
  m = s_max[0];
  for (int q = threadIdx.x; q < batch; q += blockDim.x) {
    double w = normalize ? __ddiv_rn(s_w[q], m) : s_w[q];
    if (!(w <= 1.7976931348623157e308 && w >= -1.7976931348623157e308) && v.d_flags)
      atomicOr(v.d_flags, DZ_FLAG_NONFINITE_WEIGHT);
    out.d_weights[q] = w;
    if (ex.d_w) ex.d_w[q] = (float)w;
  }
}

__global__ void uniform_sample_kernel(dz_replay_view v, dz_sample_inputs in, dz_sample_outputs out, int batch,
                                      BatchExtras ex) {
  dz::pdl_enter();
  int q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= batch) return;
  int64_t pos = in.d_rand_pos[q];
  int64_t id = v.d_ids[pos];  // replay.py:78-81
  int64_t slot = id % v.capacity;
  out.d_ids[q] = id;
  if (out.d_indices) out.d_indices[q] = pos;
  out.d_slots[q] = slot;
  if (out.d_probs) out.d_probs[q] = 0.0;
  if (out.d_weights) out.d_weights[q] = 1.0;
  emit_batch_rows(v, ex, q, slot, 1.0);
}

// ------------------------------------------------------------------------------------------------
// Gather (replay.py:718-722: get + np.stack)
// ------------------------------------------------------------------------------------------------

__global__ void __launch_bounds__(256) gather_obs_kernel(dz_replay_view v, const int64_t* __restrict__ slots,
                                                         uint8_t* __restrict__ s_tm1, uint8_t* __restrict__ s_t,
                                                         int vec16) {
  dz::pdl_enter();
  // the row index rides on grid.x (2^31 - 1 blocks); grid.y is only the <= 8-way split of one row
  const int b = blockIdx.x >> 1, which = blockIdx.x & 1;
  const uint8_t* src = v.d_obs + (slots[b] * 2 + which) * v.obs_stride;
  uint8_t* dst = (which ? s_t : s_tm1) + (int64_t)b * v.obs_bytes;
  if (vec16) {
    const int64_t nvec = v.obs_bytes >> 4;
    const uint4* s4 = reinterpret_cast<const uint4*>(src);
    uint4* d4 = reinterpret_cast<uint4*>(dst);
    for (int64_t i = blockIdx.y * (int64_t)blockDim.x + threadIdx.x; i < nvec; i += (int64_t)gridDim.y * blockDim.x)
      d4[i] = __ldg(s4 + i);
  } else {
    for (int64_t i = blockIdx.y * (int64_t)blockDim.x + threadIdx.x; i < v.obs_bytes;
         i += (int64_t)gridDim.y * blockDim.x)
      dst[i] = src[i];
  }
}

__global__ void gather_scalars_kernel(dz_replay_view v, const int64_t* __restrict__ slots, int batch, int64_t* a,
                                      double* r, double* d) {
  dz::pdl_enter();
  int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= batch) return;
  int64_t s = slots[b];
  if (a) a[b] = (int64_t)v.d_action[s];
  if (r) r[b] = v.d_reward[s];
  if (d) d[b] = v.d_discount[s];
}

// ------------------------------------------------------------------------------------------------
// Insert (replay.py:690-699) and synthetic fill
// ------------------------------------------------------------------------------------------------

__global__ void __launch_bounds__(64) apply_add_kernel(dz_replay_view v, dz_add_record rec) {
  dz::pdl_enter();
  __shared__ int64_t s_idx[2];
  __shared__ double s_val[2];
  if (threadIdx.x == 0) {
    v.d_action[rec.slot] = rec.action;
    v.d_reward[rec.slot] = rec.reward;
    v.d_discount[rec.slot] = rec.discount;
    for (int p = 0; p < rec.n_patches; ++p) {
      int64_t* dst = rec.patch_target[p] == 0 ? v.d_live : (rec.patch_target[p] == 1 ? v.d_id_at : v.d_ids);
      dst[rec.patch_pos[p]] = rec.patch_val[p];
    }
    // remove_priorities zeroes the evicted leaf (replay.py:533-534) before add_priorities sets the new one.
    s_idx[0] = rec.evict_index;
    s_val[0] = 0.0;
    s_idx[1] = rec.tree_index;
    double leaf = rec.leaf_value;
    if (rec.d_priority) {  // priority kept on the device (float32 value, widened as np.max([...]) does)
      double pr = (double)rec.d_priority[0];
      if (!finite_nonneg(pr)) {
        if (v.d_flags) atomicOr(v.d_flags, DZ_FLAG_BAD_VALUE);
        pr = 0.0;
      }
      leaf = pr == 0.0 ? 0.0 : (rec.alpha == 0.5 ? __dsqrt_rn(pr) : (rec.alpha == 1.0 ? pr : pow(pr, rec.alpha)));
    }
    s_val[1] = leaf;
  }
  __syncthreads();
  if (rec.tree_index >= 0 && v.d_tree) block_tree_set(v.d_tree, v.first_leaf, s_idx, s_val, 2);
}

__device__ __forceinline__ uint64_t mix64(uint64_t x) {
  x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
  x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
  return x ^ (x >> 31);
}

__global__ void __launch_bounds__(256) fill_obs_kernel(dz_replay_view v, int64_t row0, int64_t n, uint64_t seed) {
  dz::pdl_enter();
  const int64_t words = v.obs_bytes >> 3;
  const int64_t total = n * 2 * words;
  const uint64_t base = seed * 0x9E3779B97F4A7C15ull;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    int64_t w = i % words;
    int64_t ro = i / words;  // (row - row0)*2 + o
    int64_t row = row0 + (ro >> 1);
    int64_t o = ro & 1;
    uint64_t ctr = base + (uint64_t)(row * 2 + o) * (uint64_t)words + (uint64_t)w;
    uint64_t* dst = reinterpret_cast<uint64_t*>(v.d_obs + (row * 2 + o) * v.obs_stride) + w;
    *dst = mix64(ctr);
  }
}

__global__ void fill_scalars_kernel(dz_replay_view v, int64_t row0, int64_t n, uint64_t seed, int num_actions,
                                    double discount) {
  dz::pdl_enter();
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= n) return;
  int64_t row = row0 + i;
  const uint64_t base = seed * 0x9E3779B97F4A7C15ull + 0xD1B54A32D192ED03ull + (uint64_t)row * 4ull;
  v.d_action[row] = (int32_t)(mix64(base) % (uint64_t)num_actions);
  double u = (double)(mix64(base + 1) >> 11) * (1.0 / 9007199254740992.0);
  v.d_reward[row] = u < 0.05 ? -1.0 : (u < 0.95 ? 0.0 : 1.0);
  double u3 = (double)(mix64(base + 2) >> 11) * (1.0 / 9007199254740992.0);
  v.d_discount[row] = u3 < 0.99 ? discount : 0.0;
}

// ------------------------------------------------------------------------------------------------
// Host-side launchers shared with the learner
// ------------------------------------------------------------------------------------------------

int launch_sample(const dz_replay_view* view, int prioritized, const dz_sample_inputs* in, const dz_sample_outputs* out,
                  int batch, const BatchExtras& ex, void* stream) {
  if (batch <= 0) return fail(DZ_EINVAL, "batch must be positive");
  if (prioritized) {
    // one block: the importance weights are normalised by the batch maximum (replay.py:237-238)
    if (batch > 1024) return fail(DZ_EINVAL, "prioritized batch must be in [1,1024]");
    if (!view->d_tree || !view->d_live || !view->d_id_at) return fail(DZ_EINVAL, "prioritized view lacks tree/live/id_at");
    if (!out->d_indices || !out->d_ids || !out->d_slots || !out->d_probs || !out->d_weights)
      return fail(DZ_EINVAL, "prioritized sample needs all outputs");
    int threads = 32 * (batch < 32 ? batch : 32);
    DZ_LAUNCH(per_sample_kernel, 1, threads, batch * sizeof(double), stream, *view, *in, *out, batch, ex);
  } else {
    if (!view->d_ids) return fail(DZ_EINVAL, "uniform view lacks ids");
    DZ_LAUNCH(uniform_sample_kernel, (int)ceil_div(batch, 128), 128, 0, stream, *view, *in, *out, batch, ex);
  }
  return DZ_OK;
}

int launch_fill_scalars(const dz_replay_view* view, int64_t row0, int64_t n, uint64_t seed, int num_actions,
                        double discount, void* stream) {
  if (n <= 0) return DZ_OK;
  DZ_LAUNCH(fill_scalars_kernel, (int)ceil_div(n, 256), 256, 0, stream, *view, row0, n, seed, num_actions, discount);
  return DZ_OK;
}

int launch_update_priorities(const dz_replay_view* view, const int64_t* d_indices, const float* d_priorities, int n,
                             double alpha, int64_t size, void* stream) {
  if (n <= 32 && view->first_leaf >= 2) {
    DZ_LAUNCH(update_priorities_warp_kernel, 1, 32, 0, stream, view->d_tree, view->first_leaf, size, d_indices, d_priorities, n,
              alpha, view->d_flags);
    return DZ_OK;
  }
  for (int off = 0; off < n; off += kSetChunk) {
    int m = n - off < kSetChunk ? n - off : kSetChunk;
    DZ_LAUNCH(update_priorities_kernel, 1, 256, 0, stream, view->d_tree, view->first_leaf, size, d_indices + off,
              d_priorities + off, m, alpha, view->d_flags);
  }
  return DZ_OK;
}

}  // namespace dz

using namespace dz;

extern "C" {

const char* dz_last_error(void) { return g_last_error.c_str(); }
const char* dz_build_info(void) { return "dqn_zoo_b200 0.1 sm_100a " __DATE__ " " __TIME__; }
int64_t dz_launch_count(void) { return g_launches.load(); }

// Debug: installs (or, with nullptr, removes) the device buffer every kernel of the library stamps at its start
// (dz_common.cuh: timeline_stamp).  d_buf: >= 2 + 2 * 4000 uint64, zero-initialised by the caller.
int dz_debug_timeline(unsigned long long* d_buf) {
  DZ_CUDA_OK(cudaDeviceSynchronize());
  for (auto fn : timeline_setters())
    if (fn(d_buf) != 0) return fail(DZ_ECUDA, "dz_debug_timeline: cudaMemcpyToSymbol failed");
  return DZ_OK;
}

int dz_profile_begin(void) {
  g_profile_recs.clear();
  g_profile = true;
  return DZ_OK;
}

int dz_profile_end(char* out, int64_t cap) {
  g_profile = false;
  DZ_CUDA_OK(cudaDeviceSynchronize());
  std::map<std::string, std::pair<int64_t, double>> agg;
  std::map<std::string, ProfileRec> geo;
  std::vector<std::string> order;
  for (auto& r : g_profile_recs) {
    geo[r.name] = r;
    float ms = 0.f;
    cudaEventElapsedTime(&ms, r.a, r.b);
    cudaEventDestroy(r.a);
    cudaEventDestroy(r.b);
    if (!agg.count(r.name)) order.push_back(r.name);
    agg[r.name].first += 1;
    agg[r.name].second += ms;
  }
  g_profile_recs.clear();
  std::string js = "{";
  for (size_t i = 0; i < order.size(); ++i) {
    char buf[256];
    snprintf(buf, sizeof(buf), "%s\"%s\": [%lld, %.6f, %u, %u, %u]", i ? ", " : "", order[i].c_str(), (long long)agg[order[i]].first,
             agg[order[i]].second, geo[order[i]].gx, geo[order[i]].gy, geo[order[i]].bx);
    js += buf;
  }
  js += "}";
  if ((int64_t)js.size() + 1 > cap) return fail(DZ_EINVAL, "profile buffer too small");
  memcpy(out, js.c_str(), js.size() + 1);
  return DZ_OK;
}

int dz_sumtree_rebuild(double* d_nodes, int64_t first_leaf, int64_t n_valid, void* stream) {
  if (first_leaf <= 0 || (first_leaf & (first_leaf - 1))) return fail(DZ_EINVAL, "first_leaf must be a power of two");
  if (n_valid < 0 || n_valid > first_leaf) return fail(DZ_EINVAL, "n_valid out of range");
  int64_t tail = first_leaf - n_valid;
  DZ_LAUNCH(sumtree_zero_tail_kernel, (int)(tail > 0 ? ceil_div(tail, 256) : 1), 256, 0, stream, d_nodes, first_leaf,
            n_valid);
  int64_t width = first_leaf >> 1;
  for (; width > 1024; width >>= 1)
    DZ_LAUNCH(sumtree_level_kernel, (int)ceil_div(width, 256), 256, 0, stream, d_nodes, width);
  if (width >= 1) DZ_LAUNCH(sumtree_top_kernel, 1, 1024, 0, stream, d_nodes, width);
  return DZ_OK;
}

int dz_sumtree_set(double* d_nodes, int64_t first_leaf, int64_t size, const int64_t* d_idx, const double* d_values,
                   int64_t n, int32_t* d_flags, void* stream) {
  if (first_leaf <= 0) return fail(DZ_EINVAL, "empty tree");
  for (int64_t off = 0; off < n; off += kSetChunk) {
    int m = (int)(n - off < kSetChunk ? n - off : kSetChunk);
    DZ_LAUNCH(sumtree_set_kernel, 1, 256, 0, stream, d_nodes, first_leaf, size, d_idx + off, d_values + off, m, d_flags);
  }
  return DZ_OK;
}

int dz_sumtree_query(const double* d_nodes, int64_t first_leaf, const double* d_targets, int64_t n, int64_t* d_out_idx,
                     int32_t* d_flags, void* stream) {
  if (first_leaf <= 0) return fail(DZ_EINVAL, "empty tree");
  if (n <= 0) return DZ_OK;
  DZ_LAUNCH(sumtree_query_kernel, (int)ceil_div(n * 32, 256), 256, 0, stream, d_nodes, first_leaf, d_targets, n,
            d_out_idx, d_flags);
  return DZ_OK;
}

int dz_sumtree_get(const double* d_nodes, int64_t first_leaf, int64_t size, const int64_t* d_idx, int64_t n,
                   double* d_out, int32_t* d_flags, void* stream) {
  if (n <= 0) return DZ_OK;
  DZ_LAUNCH(sumtree_get_kernel, (int)ceil_div(n, 256), 256, 0, stream, d_nodes, first_leaf, size, d_idx, n, d_out,
            d_flags);
  return DZ_OK;
}

int dz_replay_add(const dz_replay_view* view, const dz_add_record* rec, const uint8_t* h_s_tm1, const uint8_t* h_s_t,
                  void* stream) {
  if (rec->slot < 0 || rec->slot >= view->capacity) return fail(DZ_ERANGE, "slot out of range");
  if (rec->n_patches < 0 || rec->n_patches > 4) return fail(DZ_EINVAL, "at most 4 patches");
  if (frame_store_on(view)) {   // both stacks go to the add staging area; frames_insert deduplicates their planes
    if (!h_s_tm1 || !h_s_t) return fail(DZ_EINVAL, "a frame store add needs both observations");
    int st = frames_check_add(view, rec);   // rejected before any copy or index patch is enqueued
    if (st != DZ_OK) return st;
    uint8_t* stage = view->frames.d_add_stage;
    DZ_CUDA_OK(cudaMemcpyAsync(stage, h_s_tm1, view->obs_bytes, cudaMemcpyDefault, (cudaStream_t)stream));
    DZ_CUDA_OK(cudaMemcpyAsync(stage + view->obs_stride, h_s_t, view->obs_bytes, cudaMemcpyDefault, (cudaStream_t)stream));
    DZ_LAUNCH(apply_add_kernel, 1, 64, 0, stream, *view, *rec);
    return frames_insert(view, rec, stream);
  }
  uint8_t* row = view->d_obs + rec->slot * 2 * view->obs_stride;
  // cudaMemcpyDefault: the sources may be host arrays (the reference's add path) or device buffers (frame stacks kept
  // in HBM by the device preprocessing) — the driver infers the direction from the unified address space
  if (h_s_tm1) DZ_CUDA_OK(cudaMemcpyAsync(row, h_s_tm1, view->obs_bytes, cudaMemcpyDefault, (cudaStream_t)stream));
  if (h_s_t)
    DZ_CUDA_OK(cudaMemcpyAsync(row + view->obs_stride, h_s_t, view->obs_bytes, cudaMemcpyDefault, (cudaStream_t)stream));
  DZ_LAUNCH(apply_add_kernel, 1, 64, 0, stream, *view, *rec);
  return DZ_OK;
}

int dz_replay_fill_synthetic(const dz_replay_view* view, int64_t row0, int64_t n, uint64_t seed, int32_t num_actions,
                             double discount, void* stream) {
  if (view->obs_bytes % 8) return fail(DZ_EINVAL, "obs_bytes must be a multiple of 8 for synthetic fill");
  if (row0 < 0 || row0 + n > view->capacity) return fail(DZ_ERANGE, "rows out of range");
  if (n == 0) return DZ_OK;
  int64_t total = n * 2 * (view->obs_bytes >> 3);
  int grid = (int)(ceil_div(total, 256) < 148 * 32 ? ceil_div(total, 256) : 148 * 32);
  DZ_LAUNCH(fill_obs_kernel, grid, 256, 0, stream, *view, row0, n, seed);
  DZ_LAUNCH(fill_scalars_kernel, (int)ceil_div(n, 256), 256, 0, stream, *view, row0, n, seed, num_actions, discount);
  return DZ_OK;
}

int dz_replay_sample(const dz_replay_view* view, int32_t prioritized, const dz_sample_inputs* in,
                     const dz_sample_outputs* out, int32_t batch, void* stream) {
  BatchExtras none{};
  return launch_sample(view, prioritized, in, out, batch, none, stream);
}

int dz_replay_gather(const dz_replay_view* view, const int64_t* d_slots, int32_t batch, uint8_t* d_s_tm1, uint8_t* d_s_t,
                     int64_t* d_a, double* d_r, double* d_disc, void* stream) {
  if (batch <= 0) return DZ_OK;
  if (frame_store_on(view)) {
    int st = launch_frame_assemble(view, d_slots, batch, d_s_tm1, d_s_t, view->obs_bytes, stream);
    if (st != DZ_OK) return st;
    DZ_LAUNCH(gather_scalars_kernel, (int)ceil_div(batch, 128), 128, 0, stream, *view, d_slots, batch, d_a, d_r, d_disc);
    return DZ_OK;
  }
  int vec16 = (view->obs_bytes % 16 == 0) && ((uintptr_t)d_s_tm1 % 16 == 0) && ((uintptr_t)d_s_t % 16 == 0);
  int64_t work = vec16 ? view->obs_bytes >> 4 : view->obs_bytes;
  int gx = (int)(ceil_div(work, 256) < 8 ? ceil_div(work, 256) : 8);
  dim3 grid((unsigned)batch * 2u, gx);
  DZ_LAUNCH(gather_obs_kernel, grid, 256, 0, stream, *view, d_slots, d_s_tm1, d_s_t, vec16);
  DZ_LAUNCH(gather_scalars_kernel, (int)ceil_div(batch, 128), 128, 0, stream, *view, d_slots, batch, d_a, d_r, d_disc);
  return DZ_OK;
}

int dz_replay_update_priorities(const dz_replay_view* view, const int64_t* d_indices, const float* d_priorities,
                                int32_t n, double alpha, int64_t size, void* stream) {
  if (!view->d_tree) return fail(DZ_EINVAL, "not a prioritized replay");
  return launch_update_priorities(view, d_indices, d_priorities, n, alpha, size, stream);
}

}  // extern "C"
