// Frame-deduplicated replay storage (dz_frame_store, DESIGN.md §3): insert with deduplication against a window of
// recent frames, assembly of HWC stacks from frame slots (gather and the fused learner's staging rows), and the
// closed-form synthetic fill.  The insert rule is restated in numpy by oracle/frame_store_oracle.py and compared
// with these kernels bit for bit.
#include "dz_internal.cuh"

#define DZ_TRY_F(expr) do { int _s = (expr); if (_s != DZ_OK) return _s; } while (0)

namespace dz {

__host__ __device__ __forceinline__ uint64_t frame_mix64(uint64_t x) {
  x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
  x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
  return x ^ (x >> 31);
}

// dz_frame_hash of n bytes: mix64(n ^ K0) + sum_k mix64(w_k ^ k * K1) (mod 2^64), w_k = the k-th little-endian
// 8-byte word of the bytes, zero-padded.  The sum makes it parallel; the per-word index makes it order dependent.
// A hash only selects which candidates are compared byte for byte, so collisions cost time, never correctness.
__host__ __device__ __forceinline__ uint64_t frame_hash_init(int64_t n) {
  return frame_mix64((uint64_t)n ^ 0xA0761D6478BD642Full);
}
__host__ __device__ __forceinline__ uint64_t frame_hash_word(uint64_t w, int64_t k) {
  return frame_mix64(w ^ ((uint64_t)k * 0x9E3779B97F4A7C15ull));
}

namespace {

constexpr int kW = DZ_FRAME_WINDOW;
constexpr int kMaxP = 2 * DZ_FRAME_MAX_STACK;
constexpr int kInsertThreads = 256;

__device__ __forceinline__ int64_t* window_entry(const dz_frame_store& fs, int64_t id) {
  return fs.d_state + 2 + (id % kW) * (1 + 2 * fs.stack);
}

// One add (one block): de-interleave the 2S planes of the staged s_tm1 | s_t into shared memory, hash them (one warp
// per plane), stage the window's frames (slot + hash) in shared memory, then walk the planes in order and either reuse
// a matching candidate or append at the ring head.  Every decision a plane takes is read by all threads into registers
// before a barrier, and only after that barrier does thread 0 write the shared or global state the decision read.
__global__ void __launch_bounds__(kInsertThreads) frame_insert_kernel(dz_replay_view v, dz_add_record rec) {
  dz::pdl_enter();
  const dz_frame_store fs = v.frames;
  const int S = fs.stack, P = 2 * S, nwin = kW * P;
  const int64_t fb = fs.frame_bytes, fstride = fs.frame_stride, nw = fstride >> 3, nwh = (fb + 7) >> 3;
  extern __shared__ __align__(16) uint8_t s_planes[];   // [P][frame_stride], zero padded
  __shared__ uint64_t s_hash[kMaxP];
  __shared__ int s_nonzero[kMaxP];
  __shared__ int s_wslot[kW * kMaxP];                   // window candidates in preference order (-1: none)
  __shared__ uint64_t s_whash[kW * kMaxP];
  __shared__ int s_cand[kMaxP + kW * kMaxP];
  __shared__ int s_ncand, s_choice;
  __shared__ int s_app[kMaxP];
  __shared__ uint64_t s_app_hash[kMaxP];
  __shared__ int s_row[kMaxP];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = blockDim.x >> 5;
  const int64_t ob = v.obs_bytes, id = rec.item_id;
  for (int64_t e = tid; e < 2 * ob; e += blockDim.x) {
    const int which = (int)(e / ob);
    const int64_t j = e - which * ob;
    const int c = (int)(j % S);
    s_planes[(which * S + c) * fstride + j / S] = fs.d_add_stage[which * v.obs_stride + j];
  }
  for (int64_t e = tid; e < (int64_t)P * (fstride - fb); e += blockDim.x) {
    const int p = (int)(e / (fstride - fb));
    s_planes[p * fstride + fb + e % (fstride - fb)] = 0;
  }
  // window entry e = r * P + qq: the add j = id - 1 - r (newest first), its appended slot P - 1 - qq (newest first);
  // valid while the slot still holds the frame that add appended (born == j)
  for (int e = tid; e < nwin; e += blockDim.x) {
    const int r = e / P, q = P - 1 - e % P;
    const int64_t j = id - 1 - r;
    int slot = -1;
    uint64_t h = 0;
    if (j >= 0) {
      const int64_t* ent = window_entry(fs, j);
      const int64_t sl = ent[0] == j ? ent[1 + q] : -1;
      if (sl > 0 && fs.d_frame_born[sl] == j) { slot = (int)sl; h = fs.d_frame_hash[sl]; }
    }
    s_wslot[e] = slot;
    s_whash[e] = h;
  }
  __syncthreads();
  for (int p = warp; p < P; p += nwarps) {
    const uint64_t* w = reinterpret_cast<const uint64_t*>(s_planes + p * fstride);
    uint64_t h = 0, any = 0;
    for (int64_t k = lane; k < nwh; k += 32) {
      h += frame_hash_word(w[k], k);
      any |= w[k];
    }
    for (int o = 16; o > 0; o >>= 1) {
      h += __shfl_xor_sync(0xffffffffu, h, o);
      any |= __shfl_xor_sync(0xffffffffu, any, o);
    }
    if (lane == 0) { s_hash[p] = h + frame_hash_init(fb); s_nonzero[p] = any != 0; }
  }
  __syncthreads();
  int64_t appends = fs.d_state[0];
  int n_app = 0;
  bool full = false;
  for (int p = 0; p < P; ++p) {
    // candidates whose hash matches, in preference order: appended earlier in this add (newest first), then the window
    if (warp == 0) {
      int n = 0;
      if (s_nonzero[p]) {
        const uint64_t h = s_hash[p];
        const int total = n_app + nwin;
        for (int base = 0; base < total; base += 32) {
          const int e = base + lane;
          int sl = -1;
          uint64_t hs = 0;
          if (e < n_app) { sl = s_app[n_app - 1 - e]; hs = s_app_hash[n_app - 1 - e]; }
          else if (e < total) { sl = s_wslot[e - n_app]; hs = s_whash[e - n_app]; }
          const bool m = sl > 0 && hs == h;
          const unsigned bal = __ballot_sync(0xffffffffu, m);
          if (m) s_cand[n + __popc(bal & ((1u << lane) - 1u))] = sl;
          n += __popc(bal);
        }
      }
      if (lane == 0) { s_ncand = n; s_choice = s_nonzero[p] ? -1 : 0; }
    }
    __syncthreads();
    const int ncand = s_ncand;
    const uint64_t* mine = reinterpret_cast<const uint64_t*>(s_planes + p * fstride);
    int choice = s_choice;
    for (int q = 0; q < ncand && choice < 0; ++q) {
      const uint64_t* theirs = reinterpret_cast<const uint64_t*>(fs.d_frames + s_cand[q] * fstride);
      int diff = 0;
      for (int64_t k = tid; k < nw; k += blockDim.x) diff |= theirs[k] != mine[k];
      if (!__syncthreads_or(diff)) choice = s_cand[q];   // same value in every thread
    }
    // append at the ring head, if its slot is no longer referenced by a live row
    const int64_t slot = 1 + appends % fs.num_frames;
    const bool append = choice < 0;
    full = append && appends >= fs.num_frames && fs.d_frame_last_ref[slot] >= rec.oldest_live;
    __syncthreads();                                  // every thread has read s_choice, s_cand and last_ref
    if (full) break;                                  // uniform: all threads read the same values
    if (append) {
      const uint4* src = reinterpret_cast<const uint4*>(s_planes + p * fstride);
      uint4* dst = reinterpret_cast<uint4*>(fs.d_frames + slot * fstride);
      for (int64_t k = tid; k < (fstride >> 4); k += blockDim.x) dst[k] = src[k];
      for (int e = tid; e < nwin; e += blockDim.x)   // the slot's previous frame is no longer a candidate
        if (s_wslot[e] == (int)slot) s_wslot[e] = -1;
      if (tid == 0) {
        fs.d_frame_hash[slot] = s_hash[p];
        fs.d_frame_born[slot] = id;
        s_app[n_app] = (int)slot;
        s_app_hash[n_app] = s_hash[p];
      }
      choice = (int)slot;
      ++n_app;
      ++appends;
    }
    // raised at once: a frame this row uses must not be reclaimed by a later plane of the same add
    if (tid == 0) {
      if (choice > 0) fs.d_frame_last_ref[choice] = id;
      s_row[p] = choice;
    }
    __syncthreads();
  }
  if (tid == 0) {
    int32_t* row = fs.d_row_frames + rec.slot * P;
    for (int p = 0; p < P; ++p) row[p] = full ? -1 : s_row[p];
    if (full && v.d_flags) atomicOr(v.d_flags, DZ_FLAG_FRAME_POOL_FULL);
    fs.d_state[0] = appends;
    int64_t* ent = window_entry(fs, id);
    ent[0] = id;
    for (int q = 0; q < P; ++q) ent[1 + q] = q < n_app ? s_app[q] : -1;
  }
}

// One block per (transition, s_tm1 | s_t) stack: interleaves the S planes into an HWC stack.  Slot -1 (a row the
// insert could not store) reads as zeros.
__global__ void __launch_bounds__(256) frame_assemble_kernel(dz_replay_view v, const int64_t* __restrict__ slots,
                                                             uint8_t* dst0, uint8_t* dst1, int64_t pitch, int vec) {
  dz::pdl_enter();
  const dz_frame_store fs = v.frames;
  const int S = fs.stack;
  const int b = blockIdx.x >> 1, which = blockIdx.x & 1;
  __shared__ int s_f[DZ_FRAME_MAX_STACK];
  if (threadIdx.x < S) s_f[threadIdx.x] = fs.d_row_frames[slots[b] * 2 * S + which * S + threadIdx.x];
  __syncthreads();
  uint8_t* dst = (which ? dst1 : dst0) + b * pitch;
  const int64_t fb = fs.frame_bytes;
  if (vec) {   // S == 4: four pixels of four planes -> one 16-byte store
    const uint32_t* pl[4];
#pragma unroll
    for (int c = 0; c < 4; ++c)
      pl[c] = s_f[c] < 0 ? nullptr : reinterpret_cast<const uint32_t*>(fs.d_frames + s_f[c] * fs.frame_stride);
    uint4* d4 = reinterpret_cast<uint4*>(dst);
    for (int64_t q = blockIdx.y * (int64_t)blockDim.x + threadIdx.x; q < (fb >> 2); q += (int64_t)gridDim.y * blockDim.x) {
      const uint32_t a = pl[0] ? __ldg(pl[0] + q) : 0u, bb = pl[1] ? __ldg(pl[1] + q) : 0u;
      const uint32_t c = pl[2] ? __ldg(pl[2] + q) : 0u, d = pl[3] ? __ldg(pl[3] + q) : 0u;
      const uint32_t lo_ab = __byte_perm(a, bb, 0x5140), lo_cd = __byte_perm(c, d, 0x5140);
      const uint32_t hi_ab = __byte_perm(a, bb, 0x7362), hi_cd = __byte_perm(c, d, 0x7362);
      d4[q] = make_uint4(__byte_perm(lo_ab, lo_cd, 0x5410), __byte_perm(lo_ab, lo_cd, 0x7632),
                         __byte_perm(hi_ab, hi_cd, 0x5410), __byte_perm(hi_ab, hi_cd, 0x7632));
    }
  } else {
    for (int64_t j = blockIdx.y * (int64_t)blockDim.x + threadIdx.x; j < fb * S; j += (int64_t)gridDim.y * blockDim.x) {
      const int f = s_f[j % S];
      dst[j] = f < 0 ? 0 : fs.d_frames[f * fs.frame_stride + j / S];
    }
  }
}

// ---- closed-form synthetic fill ---------------------------------------------------------------------------------
// Transition i is step t = i % L of episode e = i / L; frame j (0..T_e) of episode e is append a = e (L + 1) + j and
// lives in slot 1 + a.  T_e = min(L, n - e L) transitions are in episode e.
struct SynthGeom {
  int64_t n, L;
  __device__ int64_t episode_len(int64_t e) const { return min(L, n - e * L); }
};

__global__ void __launch_bounds__(256) frame_fill_frames_kernel(dz_replay_view v, SynthGeom g, int64_t appends,
                                                                uint64_t seed) {
  dz::pdl_enter();
  const dz_frame_store fs = v.frames;
  const int lane = threadIdx.x & 31;
  const int64_t a = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
  if (a >= appends) return;
  const int64_t words = fs.frame_bytes >> 3, slot = 1 + a;
  const uint64_t base = seed * 0x9E3779B97F4A7C15ull + 0x5851F42D4C957F2Dull + (uint64_t)a * (uint64_t)words;
  uint64_t* dst = reinterpret_cast<uint64_t*>(fs.d_frames + slot * fs.frame_stride);
  uint64_t h = 0;
  for (int64_t k = lane; k < fs.frame_stride >> 3; k += 32) {
    const uint64_t w = k < words ? frame_mix64(base + (uint64_t)k) : 0ull;
    dst[k] = w;
    if (k < words) h += frame_hash_word(w, k);
  }
  for (int o = 16; o > 0; o >>= 1) h += __shfl_xor_sync(0xffffffffu, h, o);
  if (lane == 0) {
    const int64_t e = a / (g.L + 1), j = a % (g.L + 1), id0 = e * g.L;
    fs.d_frame_hash[slot] = h + frame_hash_init(fs.frame_bytes);
    fs.d_frame_born[slot] = id0 + (j > 0 ? j - 1 : 0);
    fs.d_frame_last_ref[slot] = id0 + min(j + fs.stack - 1, g.episode_len(e) - 1);
  }
}

__device__ __forceinline__ int32_t synth_slot(const SynthGeom& g, int S, int64_t i, int which, int c) {
  const int64_t e = i / g.L, t = i % g.L + which;   // stack index within the episode
  int64_t j;
  if (t < S) {
    if (c > t) return 0;
    j = c;
  } else {
    j = t - S + 1 + c;
  }
  return (int32_t)(1 + e * (g.L + 1) + j);
}

__global__ void frame_fill_rows_kernel(dz_replay_view v, SynthGeom g) {
  dz::pdl_enter();
  const int S = v.frames.stack, P = 2 * S;
  const int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (k >= g.n * P) return;
  const int64_t i = k / P;
  const int p = (int)(k % P);
  v.frames.d_row_frames[k] = synth_slot(g, S, i, p / S, p % S);
}

__global__ void frame_fill_state_kernel(dz_replay_view v, SynthGeom g, int64_t appends) {
  dz::pdl_enter();
  const dz_frame_store fs = v.frames;
  const int P = 2 * fs.stack;
  const int r = threadIdx.x;   // window entry
  if (r >= kW) return;
  int64_t* ent = fs.d_state + 2 + r * (1 + P);
  for (int q = 0; q <= P; ++q) ent[q] = -1;
  // the add of id i wrote entry i % kW; the newest such id with i < n
  const int64_t last = g.n - 1;
  const int64_t i = last - ((last - r) % kW + kW) % kW;
  if (i >= 0 && i > last - kW) {
    const int64_t e = i / g.L, t = i % g.L, a0 = e * (g.L + 1);
    ent[0] = i;
    if (t == 0) { ent[1] = 1 + a0; ent[2] = 2 + a0; }
    else ent[1] = 1 + a0 + t + 1;
  }
  if (r == 0) { fs.d_state[0] = appends; fs.d_state[1] = 0; }
}

}  // namespace

bool frame_store_on(const dz_replay_view* v) { return v->frames.d_frames != nullptr; }

int frames_check(const dz_replay_view* v) {
  const dz_frame_store& fs = v->frames;
  if (fs.stack < 1 || fs.stack > DZ_FRAME_MAX_STACK) return fail(DZ_EINVAL, "frame store stack depth must be in [1, 8]");
  if (fs.num_frames < 1 || fs.frame_bytes < 1 || fs.frame_stride % 16 || fs.frame_stride < fs.frame_bytes)
    return fail(DZ_EINVAL, "bad frame store geometry");
  if (v->obs_bytes != fs.frame_bytes * fs.stack) return fail(DZ_EINVAL, "obs_bytes != frame_bytes * stack");
  if (!fs.d_row_frames || !fs.d_frame_hash || !fs.d_frame_born || !fs.d_frame_last_ref || !fs.d_state || !fs.d_add_stage)
    return fail(DZ_EINVAL, "frame store lacks a buffer");
  return DZ_OK;
}

int frames_check_add(const dz_replay_view* v, const dz_add_record* rec) {
  DZ_TRY_F(frames_check(v));
  if (rec->item_id < 0 || rec->oldest_live < 0 || rec->oldest_live > rec->item_id)
    return fail(DZ_EINVAL, "frame store add needs 0 <= oldest_live <= item_id");
  if (2 * v->frames.stack * v->frames.frame_stride > DZ_FRAME_MAX_STAGE_BYTES)
    return fail(DZ_EINVAL, "frame store: 2 * stack * frame_stride must be <= DZ_FRAME_MAX_STAGE_BYTES");
  return DZ_OK;
}

int frames_insert(const dz_replay_view* v, const dz_add_record* rec, void* stream) {
  DZ_TRY_F(frames_check_add(v, rec));
  const int64_t smem = 2 * v->frames.stack * v->frames.frame_stride;
  static bool attr_done = false;
  if (!attr_done) {
    DZ_CUDA_OK(cudaFuncSetAttribute(frame_insert_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    DZ_FRAME_MAX_STAGE_BYTES));
    attr_done = true;
  }
  DZ_LAUNCH(frame_insert_kernel, 1, kInsertThreads, smem, stream, *v, *rec);
  return DZ_OK;
}

int launch_frame_assemble(const dz_replay_view* v, const int64_t* d_slots, int batch, uint8_t* dst0, uint8_t* dst1,
                          int64_t pitch, void* stream) {
  DZ_TRY_F(frames_check(v));
  if (batch <= 0) return DZ_OK;
  const dz_frame_store& fs = v->frames;
  const int vec = fs.stack == 4 && fs.frame_bytes % 4 == 0 && pitch % 16 == 0 && (uintptr_t)dst0 % 16 == 0 &&
                  (uintptr_t)dst1 % 16 == 0;
  const int64_t work = vec ? fs.frame_bytes >> 2 : fs.frame_bytes * fs.stack;
  const int gy = (int)(ceil_div(work, 256) < 8 ? ceil_div(work, 256) : 8);
  dim3 grid((unsigned)batch * 2u, gy);
  DZ_LAUNCH(frame_assemble_kernel, grid, 256, 0, stream, *v, d_slots, dst0, dst1, pitch, vec);
  return DZ_OK;
}

}  // namespace dz

using namespace dz;

extern "C" {

int dz_replay_fill_synthetic_frames(const dz_replay_view* view, int64_t n, int64_t episode_length, uint64_t seed,
                                    int32_t num_actions, double discount, void* stream) {
  if (!frame_store_on(view)) return fail(DZ_EINVAL, "not a frame store");
  DZ_TRY_F(frames_check(view));
  if (view->frames.frame_bytes % 8) return fail(DZ_EINVAL, "frame_bytes must be a multiple of 8 for synthetic fill");
  if (episode_length < 1) return fail(DZ_EINVAL, "episode_length must be positive");
  if (n < 0 || n > view->capacity) return fail(DZ_ERANGE, "rows out of range");
  if (n == 0) return DZ_OK;
  const int64_t appends = n + ceil_div(n, episode_length);
  if (appends > view->frames.num_frames) return fail(DZ_EINVAL, "frame_capacity is too small for the synthetic fill");
  SynthGeom g{n, episode_length};
  DZ_LAUNCH(frame_fill_frames_kernel, (unsigned)ceil_div(appends * 32, 256), 256, 0, stream, *view, g, appends, seed);
  DZ_LAUNCH(frame_fill_rows_kernel, (unsigned)ceil_div(n * 2 * view->frames.stack, 256), 256, 0, stream, *view, g);
  DZ_LAUNCH(frame_fill_state_kernel, 1, 32, 0, stream, *view, g, appends);
  return launch_fill_scalars(view, 0, n, seed, num_actions, discount, stream);
}

int dz_test_frame_hash(const uint8_t* h_bytes, int64_t n, uint64_t* out) {
  uint64_t h = frame_hash_init(n);
  for (int64_t k = 0; k * 8 < n; ++k) {
    uint64_t w = 0;
    for (int b = 0; b < 8 && k * 8 + b < n; ++b) w |= (uint64_t)h_bytes[k * 8 + b] << (8 * b);
    h += frame_hash_word(w, k);
  }
  *out = h;
  return DZ_OK;
}

}  // extern "C"
