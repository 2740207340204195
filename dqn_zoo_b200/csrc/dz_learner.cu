// Learner half of the hot path: the jitted `update` of every dqn_zoo agent as hand-written CUDA.
//
//   networks      networks.py:58-363   (Nature-CNN torso, DQN / C51 / QR / IQN / Rainbow heads)
//   loss_fn       dqn/agent.py:85-107, double_q/agent.py:85-111, prioritized/agent.py:86-113,
//                 c51/agent.py:87-107, qrdqn/agent.py:88-110, rainbow/agent.py:85-109, iqn/agent.py:178-214
//   rlax 0.1.2    q_learning, double_q_learning, clip_gradient, l2_loss, categorical_l2_project,
//                 categorical_[double_]q_learning, quantile_q_learning (restated; SURVEY §8(c))
//   optax 0.1.2   adam, rmsprop(centered), clip_by_global_norm, apply_updates
//   _learn glue   rainbow/agent.py:181-198, prioritized/agent.py:187-206
//
// Gradients flow only through online(s_tm1).  All forward passes of a layer are one grouped
// launch (dz_gemm.cuh); the replay gather is fused into conv1's operand load.
#include <algorithm>
#include <cmath>
#include <map>
#include <vector>

#include "dz_gemm.cuh"
#include "dz_tc.cuh"
#include "dz_internal.cuh"
#include "dz_umma_net.cuh"

namespace dz {

// ------------------------------------------------------------------------------------------------
// Parameter layout (canonical names; haiku layouts) — must match oracle/learner_oracle.py:param_shapes
// ------------------------------------------------------------------------------------------------

struct TensorInfo {
  std::string name;
  int64_t shape[4];
  int ndim;
  int64_t offset, count;
};

struct Dims {
  int H, W, C;       // observation
  int h1, w1, h2, w2, h3, w3;
  int feat;          // h3*w3*64
  int out;           // head outputs (family dependent)
};

static inline int conv_out(int n, int k, int s) { return (n - k) / s + 1; }

static Dims make_dims(const dz_learner_config& c) {
  Dims d;
  d.H = c.obs_h; d.W = c.obs_w; d.C = c.obs_c;
  d.h1 = conv_out(d.H, 8, 4); d.w1 = conv_out(d.W, 8, 4);
  d.h2 = conv_out(d.h1, 4, 2); d.w2 = conv_out(d.w1, 4, 2);
  d.h3 = conv_out(d.h2, 3, 1); d.w3 = conv_out(d.w2, 3, 1);
  d.feat = d.h3 * d.w3 * 64;
  switch (c.kind) {
    case DZ_C51: d.out = c.num_actions * c.num_atoms; break;
    case DZ_QRDQN: d.out = c.num_quantiles * c.num_actions; break;
    case DZ_RAINBOW: d.out = c.num_actions * c.num_atoms; break;
    default: d.out = c.num_actions;
  }
  return d;
}

struct Layout {
  std::vector<TensorInfo> t;
  std::map<std::string, int> index;
  int64_t total = 0;
  void add(const std::string& name, std::initializer_list<int64_t> shape) {
    TensorInfo ti;
    ti.name = name;
    ti.ndim = (int)shape.size();
    ti.count = 1;
    int i = 0;
    for (auto s : shape) { ti.shape[i++] = s; ti.count *= s; }
    for (; i < 4; ++i) ti.shape[i] = 1;
    ti.offset = total;
    total += (ti.count + 3) / 4 * 4;  // keep every tensor 16-byte aligned for float4 loads
    index[name] = (int)t.size();
    t.push_back(ti);
  }
  int64_t off(const std::string& name) const { return t[index.at(name)].offset; }
  bool has(const std::string& name) const { return index.count(name) != 0; }
};

static Layout make_layout(const dz_learner_config& c) {
  Layout L;
  Dims d = make_dims(c);
  L.add("conv1/w", {8, 8, d.C, 32}); L.add("conv1/b", {32});
  L.add("conv2/w", {4, 4, 32, 64});  L.add("conv2/b", {64});
  L.add("conv3/w", {3, 3, 64, 64});  L.add("conv3/b", {64});
  if (c.kind == DZ_RAINBOW) {
    const char* streams[2] = {"adv", "val"};
    for (int s = 0; s < 2; ++s) {
      std::string p = streams[s];
      int64_t n_out = s == 0 ? (int64_t)c.num_actions * c.num_atoms : c.num_atoms;
      L.add(p + "1/mu/w", {d.feat, 512}); L.add(p + "1/mu/b", {512});
      L.add(p + "1/sigma/w", {d.feat, 512}); L.add(p + "1/sigma/b", {512});
      L.add(p + "2/mu/w", {512, n_out}); L.add(p + "2/sigma/w", {512, n_out}); L.add(p + "2/sigma/b", {n_out});
    }
    return L;
  }
  if (c.kind == DZ_IQN) { L.add("embed/w", {c.latent_dim, d.feat}); L.add("embed/b", {d.feat}); }
  L.add("fc1/w", {d.feat, 512}); L.add("fc1/b", {512});
  L.add("head/w", {512, d.out});
  bool shared = c.kind == DZ_DOUBLE_Q || c.kind == DZ_PRIORITIZED;
  L.add("head/b", {shared ? 1 : d.out});
  return L;
}

struct Bump {
  char* base;
  int64_t used = 0;
  template <typename T> T* take(int64_t n) {
    int64_t bytes = (n * (int64_t)sizeof(T) + 255) / 256 * 256;
    T* p = base ? reinterpret_cast<T*>(base + used) : nullptr;
    used += bytes;
    return p;
  }
};

static int validate(const dz_learner_config& c) {
  if (c.kind < 0 || c.kind > DZ_IQN) return fail(DZ_EINVAL, "unknown agent kind");
  if (c.batch <= 0 || c.batch > 1024) return fail(DZ_EINVAL, "batch must be in [1,1024]");
  if (c.obs_c != 4) return fail(DZ_EINVAL, "obs_c must be 4 (stacked frames; conv1 reads uchar4 pixels)");
  if (c.obs_w % 4) return fail(DZ_EINVAL, "obs_w must be a multiple of 4");
  if (c.obs_h < 36 || c.obs_w < 36) return fail(DZ_EINVAL, "observation too small for the Nature-CNN torso");
  if (c.num_actions <= 0 || c.num_actions > 64) return fail(DZ_EINVAL, "num_actions must be in [1,64]");
  if ((c.kind == DZ_C51 || c.kind == DZ_RAINBOW) && (c.num_atoms < 2 || c.num_atoms > 128)) return fail(DZ_EINVAL, "num_atoms must be in [2,128]");
  if (c.kind == DZ_QRDQN && (c.num_quantiles < 1 || c.num_quantiles > 256)) return fail(DZ_EINVAL, "num_quantiles must be in [1,256]");
  if (c.kind == DZ_IQN) {
    if (c.latent_dim <= 0 || c.latent_dim % 16) return fail(DZ_EINVAL, "latent_dim must be a positive multiple of 16");
    int mx = c.tau_samples_s_tm1 > c.tau_samples_s_t ? c.tau_samples_s_tm1 : c.tau_samples_s_t;
    mx = mx > c.tau_samples_policy ? mx : c.tau_samples_policy;
    if (c.tau_samples_s_tm1 <= 0 || c.tau_samples_s_t <= 0 || c.tau_samples_policy <= 0 || mx > 256)
      return fail(DZ_EINVAL, "tau sample counts must be in [1,256]");
  }
  return DZ_OK;
}

}  // namespace dz

using namespace dz;

// ------------------------------------------------------------------------------------------------
// Small kernels
// ------------------------------------------------------------------------------------------------

namespace {

struct FinishNN {  // split-K partials of an NN problem -> bias / noisy combine / relu
  const float* partial; int splits; long long stride; int M, N; int dual;
  const float* bias; const float* bias2; const float* c_scale; int relu; int bias_shared; float* out;
};
struct FinishNNBatch { FinishNN f[kMaxProblems]; int n; };

__global__ void __launch_bounds__(256) finish_nn_kernel(const __grid_constant__ FinishNNBatch b) {
  dz::pdl_enter();
  const FinishNN& f = b.f[blockIdx.y];
  long long total = (long long)f.M * f.N;
  if ((f.N & 3) == 0 && ((reinterpret_cast<uintptr_t>(f.partial) | reinterpret_cast<uintptr_t>(f.out) | (uintptr_t)(f.stride * 4)) & 15) == 0) {
    // 16-byte path (every layer except the odd-width heads): same per-element order of additions
    const long long total4 = total >> 2;
    for (long long i4 = blockIdx.x * (long long)blockDim.x + threadIdx.x; i4 < total4; i4 += (long long)gridDim.x * blockDim.x) {
      const long long i = i4 << 2;
      const int n = (int)(i % f.N);
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      for (int k = 0; k < f.splits; ++k) {
        const float4 x = *reinterpret_cast<const float4*>(f.partial + k * f.stride + i);
        v.x += x.x; v.y += x.y; v.z += x.z; v.w += x.w;
      }
      if (f.bias) {
        if (f.bias_shared) { const float s = f.bias[0]; v.x += s; v.y += s; v.z += s; v.w += s; }
        else { v.x += f.bias[n]; v.y += f.bias[n + 1]; v.z += f.bias[n + 2]; v.w += f.bias[n + 3]; }
      }
      if (f.dual && f.bias2) {
        v.x = fmaf(f.bias2[n], f.c_scale[n], v.x); v.y = fmaf(f.bias2[n + 1], f.c_scale[n + 1], v.y);
        v.z = fmaf(f.bias2[n + 2], f.c_scale[n + 2], v.z); v.w = fmaf(f.bias2[n + 3], f.c_scale[n + 3], v.w);
      }
      if (f.relu) { v.x = fmaxf(v.x, 0.f); v.y = fmaxf(v.y, 0.f); v.z = fmaxf(v.z, 0.f); v.w = fmaxf(v.w, 0.f); }
      *reinterpret_cast<float4*>(f.out + i) = v;
    }
    return;
  }
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    int n = (int)(i % f.N);
    float v = 0.f;
    for (int k = 0; k < f.splits; ++k) v += f.partial[k * f.stride + i];
    if (f.bias) v += f.bias_shared ? f.bias[0] : f.bias[n];
    if (f.dual && f.bias2) v = fmaf(f.bias2[n], f.c_scale[n], v);   // sigma bias of the noisy layer
    if (f.relu) v = fmaxf(v, 0.f);
    f.out[i] = v;
  }
}

struct FinishTN {  // split partials [Kext][N] of a TN problem -> weight / bias gradients
  const float* partial; int splits; long long stride; int K, N;
  float* C; float* C2; float* Cb; float* Cb2; const float* a_scale; const float* c_scale;
};
struct FinishTNBatch { FinishTN f[kMaxProblems]; int n; };

__global__ void __launch_bounds__(256) finish_tn_kernel(const __grid_constant__ FinishTNBatch b) {
  dz::pdl_enter();
  const FinishTN& f = b.f[blockIdx.y];
  int Kext = f.K + ((f.Cb || f.Cb2) ? 1 : 0);
  long long total = (long long)Kext * f.N;
  if ((f.N & 3) == 0 && !f.C2 && !f.Cb2 && f.C &&
      ((reinterpret_cast<uintptr_t>(f.partial) | reinterpret_cast<uintptr_t>(f.C) | reinterpret_cast<uintptr_t>(f.Cb) | (uintptr_t)(f.stride * 4)) & 15) == 0) {
    const long long total4 = total >> 2;
    for (long long i4 = blockIdx.x * (long long)blockDim.x + threadIdx.x; i4 < total4; i4 += (long long)gridDim.x * blockDim.x) {
      const long long i = i4 << 2;
      const int k = (int)(i / f.N), n = (int)(i % f.N);
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      for (int s = 0; s < f.splits; ++s) {
        const float4 x = *reinterpret_cast<const float4*>(f.partial + s * f.stride + i);
        v.x += x.x; v.y += x.y; v.z += x.z; v.w += x.w;
      }
      if (k < f.K) *reinterpret_cast<float4*>(f.C + i) = v;
      else if (f.Cb) *reinterpret_cast<float4*>(f.Cb + n) = v;
    }
    return;
  }
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    int k = (int)(i / f.N), n = (int)(i % f.N);
    float v = 0.f;
    for (int s = 0; s < f.splits; ++s) v += f.partial[s * f.stride + i];
    if (k < f.K) {
      if (f.C) f.C[i] = v;
      if (f.C2) f.C2[i] = v * f.a_scale[k] * f.c_scale[n];
    } else {
      if (f.Cb) f.Cb[n] = v;
      if (f.Cb2) f.Cb2[n] = v * f.c_scale[n];
    }
  }
}

struct FinishNT {  // split partials [M][K] (+ dual second half) of up to two NT problems -> summed, masked output
  const float* partial[2]; const float* a_scale[2]; int nsrc; int splits; long long stride; int M, K; int dual;
  const float* mask; float* out;
  float* out_hi; float* out_lo;   // optional: the tf32 hi/lo pair the tcgen05 kernels read (saves a separate split launch)
};
struct FinishNTBatch { FinishNT f[2]; };   // blockIdx.y selects the job

__global__ void __launch_bounds__(256) finish_nt_kernel(const __grid_constant__ FinishNTBatch fb) {
  dz::pdl_enter();
  const FinishNT& f = fb.f[blockIdx.y];
  long long total = (long long)f.M * f.K;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    float v = 0.f;
    for (int q = 0; q < f.nsrc; ++q) {
      float a = 0.f;
      for (int s = 0; s < f.splits; ++s) a += f.partial[q][s * f.stride + i];
      v += a;
    }
    if (f.mask && !(f.mask[i] > 0.f)) v = 0.f;
    f.out[i] = v;
    if (f.out_hi) {
      const float h = tc::rn_tf32(v);
      f.out_hi[i] = h;
      f.out_lo[i] = tc::rn_tf32(v - h);
    }
  }
}

// col2im for the conv input gradient: dX[b,y,x,c] = sum over kernel taps of dcol, times ReLU mask.
__global__ void __launch_bounds__(256) col2im_kernel(const float* __restrict__ dcol, const float* __restrict__ act,
                                                     float* __restrict__ dx, int nimg, int H, int W, int Cin, int KH, int KW,
                                                     int S, int OH, int OW) {
  dz::pdl_enter();
  long long total = (long long)nimg * H * W * Cin;
  const int K = KH * KW * Cin;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    int c = (int)(i % Cin);
    long long t = i / Cin;
    int x = (int)(t % W); t /= W;
    int y = (int)(t % H);
    int b = (int)(t / H);
    float v = 0.f;
    if (act[i] > 0.f) {
      for (int kh = 0; kh < KH; ++kh) {
        int yy = y - kh;
        if (yy < 0 || yy % S) continue;
        int oy = yy / S;
        if (oy >= OH) continue;
        for (int kw = 0; kw < KW; ++kw) {
          int xx = x - kw;
          if (xx < 0 || xx % S) continue;
          int ox = xx / S;
          if (ox >= OW) continue;
          v += dcol[((long long)(b * OH + oy) * OW + ox) * K + (kh * KW + kw) * Cin + c];
        }
      }
    }
    dx[i] = v;
  }
}

__global__ void add_mask_kernel(const float* __restrict__ a, const float* __restrict__ b, const float* __restrict__ act,
                                float* __restrict__ out, long long n) {
  dz::pdl_enter();
  long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i < n) out[i] = act[i] > 0.f ? a[i] + b[i] : 0.f;
}

__global__ void sum_to_scalar_kernel(const float* __restrict__ v, int n, float* out) {
  dz::pdl_enter();
  __shared__ float s[32];
  float acc = 0.f;
  for (int i = threadIdx.x; i < n; i += blockDim.x) acc += v[i];
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0) s[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x < 32) {
    acc = threadIdx.x < (blockDim.x >> 5) ? s[threadIdx.x] : 0.f;
    acc = warp_sum(acc);
    if (threadIdx.x == 0) out[0] = acc;
  }
}

// ---- IQN helpers -------------------------------------------------------------------------------

// IQN value head at training size (networks.py:285-287): out[m, a] = sum_k h1[m, k] W[k, a] + b[a] with
// M = batch * tau_samples rows (thousands), K = 512 and only num_actions (<= 18) columns.  A tiled GEMM wastes its
// N tile here; instead one warp owns one row: coalesced float4 reads of the row, W^T resident in shared memory,
// A warp reductions.  Up to three applies (blockIdx.y) per launch.
constexpr int kSkinnyMaxN = 18;
struct SkinnyHead { const float* A[3]; const float* W[3]; const float* bias[3]; float* out[3]; int M[3]; int n; };

__global__ void __launch_bounds__(256) iqn_head_fwd_kernel(const __grid_constant__ SkinnyHead h, int N) {
  dz::pdl_enter();
  constexpr int K = 512;
  __shared__ __align__(16) float Ws[kSkinnyMaxN * K];
  const int q = blockIdx.y;
  const float* __restrict__ W = h.W[q];
  for (int i = threadIdx.x; i < K * N; i += 256) {      // W is [K][N]: transpose into Ws[n][k]
    int k = i / N, n = i - k * N;
    Ws[n * K + k] = W[i];
  }
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int m = blockIdx.x * 8 + warp; m < h.M[q]; m += gridDim.x * 8) {
    const float4* a4 = reinterpret_cast<const float4*>(h.A[q] + (long long)m * K);
    float4 a[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) a[i] = a4[lane + 32 * i];
    float mine = 0.f;
    for (int n = 0; n < N; ++n) {
      const float4* w4 = reinterpret_cast<const float4*>(Ws + n * K);
      float acc = 0.f;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float4 w = w4[lane + 32 * i];
        acc = fmaf(a[i].x, w.x, acc); acc = fmaf(a[i].y, w.y, acc); acc = fmaf(a[i].z, w.z, acc); acc = fmaf(a[i].w, w.w, acc);
      }
      acc = warp_sum(acc);
      if (lane == n) mine = acc;
    }
    if (lane < N) h.out[q][(long long)m * N + lane] = mine + h.bias[q][lane];
  }
}

// Input gradient of the same head: dh1[m, k] = [h1 > 0] * sum_a dout[m, a] W[k, a]  (one thread = 4 consecutive k).
__global__ void __launch_bounds__(256) iqn_head_dgrad_kernel(const float* __restrict__ dout, const float* __restrict__ W,
                                                             const float* __restrict__ h1, float* __restrict__ dh1, int M, int N) {
  dz::pdl_enter();
  constexpr int K = 512;
  __shared__ float Ws[K * kSkinnyMaxN];
  for (int i = threadIdx.x; i < K * N; i += 256) Ws[i] = W[i];
  __syncthreads();
  const long long total = (long long)M * (K / 4);
  for (long long i = blockIdx.x * 256LL + threadIdx.x; i < total; i += (long long)gridDim.x * 256) {
    const int m = (int)(i >> 7), k = (int)(i & 127) * 4;
    float d[kSkinnyMaxN];
    for (int n = 0; n < N; ++n) d[n] = dout[(long long)m * N + n];
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int n = 0; n < N; ++n) {
      v.x = fmaf(d[n], Ws[(k + 0) * N + n], v.x);
      v.y = fmaf(d[n], Ws[(k + 1) * N + n], v.y);
      v.z = fmaf(d[n], Ws[(k + 2) * N + n], v.z);
      v.w = fmaf(d[n], Ws[(k + 3) * N + n], v.w);
    }
    const float4 h = *reinterpret_cast<const float4*>(h1 + (long long)m * K + k);
    v.x = h.x > 0.f ? v.x : 0.f; v.y = h.y > 0.f ? v.y : 0.f; v.z = h.z > 0.f ? v.z : 0.f; v.w = h.w > 0.f ? v.w : 0.f;
    *reinterpret_cast<float4*>(dh1 + (long long)m * K + k) = v;
  }
}

// cos(pi * i * tau), i = 1..latent; the product is formed in float32 as in networks.py:277-278.
__global__ void iqn_cos_kernel(const float* __restrict__ taus, float* __restrict__ out, long long rows, int latent) {
  dz::pdl_enter();
  long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= rows * latent) return;
  int j = (int)(i % latent);
  float pim = __fmul_rn((float)(j + 1), 3.14159274101257324f);
  out[i] = cosf(__fmul_rn(pim, taus[i / latent]));
}

// dE = dHI * F * (E > 0) in place; dF[b,k] = sum_n dHI[b,n,k] * E[b,n,k]; dfeat masked by act3 > 0.
__global__ void __launch_bounds__(256) iqn_hadamard_bwd_kernel(float* __restrict__ dHI, const float* __restrict__ E,
                                                               const float* __restrict__ F, float* __restrict__ dfeat,
                                                               int B, int N, int D) {
  dz::pdl_enter();
  long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= (long long)B * D) return;
  int b = (int)(i / D), k = (int)(i % D);
  float f = F[i], acc = 0.f;
  for (int n = 0; n < N; ++n) {
    long long j = ((long long)b * N + n) * D + k;
    float g = dHI[j], e = E[j];
    acc += g * e;
    dHI[j] = e > 0.f ? g * f : 0.f;
  }
  dfeat[i] = f > 0.f ? acc : 0.f;  // F is the post-ReLU conv3 output: mask for the conv3 pre-activation
}

// Packed variant for the tcgen05 path: same math, but dE is written ONLY as the hi/lo TF32 tile images of the
// transposed operand (rows k, reduction m = b*N + n; layout in dz_tcp.cuh) that the embedding weight-gradient GEMM
// consumes.  One block = one sample b x 64 features; requires N == 64 and D % 64 == 0.
__global__ void __launch_bounds__(256) iqn_hadamard_bwd_packed_kernel(const float* __restrict__ dHI, const float* __restrict__ E,
                                                                      const float* __restrict__ F, float* __restrict__ dfeat,
                                                                      float* __restrict__ img_hi, float* __restrict__ img_lo,
                                                                      int rg_total, int D) {
  dz::pdl_enter();
  constexpr int N = 64;
  __shared__ float tile[64][65];
  __shared__ float red[16][64];
  const int b = blockIdx.y, k0 = blockIdx.x * 64, tid = threadIdx.x;
  const int a = tid >> 4, k4 = (tid & 15) * 4;
  const float4 f = *reinterpret_cast<const float4*>(F + (long long)b * D + k0 + k4);
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    const int n = a + 16 * q;
    const long long j = ((long long)b * N + n) * D + k0 + k4;
    const float4 g = *reinterpret_cast<const float4*>(dHI + j);
    const float4 e = *reinterpret_cast<const float4*>(E + j);
    acc.x = fmaf(g.x, e.x, acc.x); acc.y = fmaf(g.y, e.y, acc.y); acc.z = fmaf(g.z, e.z, acc.z); acc.w = fmaf(g.w, e.w, acc.w);
    tile[n][k4 + 0] = e.x > 0.f ? g.x * f.x : 0.f;
    tile[n][k4 + 1] = e.y > 0.f ? g.y * f.y : 0.f;
    tile[n][k4 + 2] = e.z > 0.f ? g.z * f.z : 0.f;
    tile[n][k4 + 3] = e.w > 0.f ? g.w * f.w : 0.f;
  }
  red[a][k4 + 0] = acc.x; red[a][k4 + 1] = acc.y; red[a][k4 + 2] = acc.z; red[a][k4 + 3] = acc.w;
  __syncthreads();
  if (tid < 64) {
    float sum = 0.f;
#pragma unroll
    for (int r = 0; r < 16; ++r) sum += red[r][tid];
    const long long i = (long long)b * D + k0 + tid;
    dfeat[i] = F[i] > 0.f ? sum : 0.f;   // F is the post-ReLU conv3 output: mask for the conv3 pre-activation
  }
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    const int id = tid + q * 256;
    const int r = id & 7, c = (id >> 3) & 3, rg = (id >> 5) & 7, kb = id >> 8;
    const int k = k0 + rg * 8 + r, ml = kb * 16 + c * 4;
    float4 x = make_float4(tile[ml][rg * 8 + r], tile[ml + 1][rg * 8 + r], tile[ml + 2][rg * 8 + r], tile[ml + 3][rg * 8 + r]);
    float4 h, l;
    h.x = tc::rn_tf32(x.x); l.x = tc::rn_tf32(x.x - h.x);
    h.y = tc::rn_tf32(x.y); l.y = tc::rn_tf32(x.y - h.y);
    h.z = tc::rn_tf32(x.z); l.z = tc::rn_tf32(x.z - h.z);
    h.w = tc::rn_tf32(x.w); l.w = tc::rn_tf32(x.w - h.w);
    const long long off = (((((long long)(b * 4 + kb) * rg_total + (k >> 3)) << 2) + c) << 5) + (k & 7) * 4;
    *reinterpret_cast<float4*>(img_hi + off) = h;
    *reinterpret_cast<float4*>(img_lo + off) = l;
  }
}

// ---- randomness --------------------------------------------------------------------------------

__device__ __forceinline__ void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1,
                                              uint32_t out[4]) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
    uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
    uint32_t n0 = hi1 ^ c1 ^ k0, n1 = lo1, n2 = hi0 ^ c3 ^ k1, n3 = lo0;
    c0 = n0; c1 = n1; c2 = n2; c3 = n3;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

// kind 0: U[0,1) (IQN taus); kind 1: sign(n)*sqrt|n|, n ~ TruncNormal(-2,2) (networks.py:142-144).
__global__ void randomness_kernel(float* __restrict__ out, long long n, uint64_t seed, const int64_t* counters, int kind,
                                  uint32_t stream_id) {
  dz::pdl_enter();
  long long i4 = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i4 * 4 >= n) return;
  uint64_t ctr = (uint64_t)counters[1];
  uint32_t r[4];
  philox4x32_10((uint32_t)i4, (uint32_t)(i4 >> 32), (uint32_t)ctr, (uint32_t)(ctr >> 32) ^ (stream_id << 24), (uint32_t)seed,
                (uint32_t)(seed >> 32), r);
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    long long i = i4 * 4 + j;
    if (i >= n) break;
    float u = (float)(r[j] >> 8) * (1.0f / 16777216.0f);  // [0,1)
    if (kind == 0) {
      out[i] = u;
    } else {
      const float lo = -0.95449973610364158f;  // erf(-2/sqrt(2))
      float v = lo + (-2.0f * lo) * ((float)(r[j] >> 8) + 0.5f) * (1.0f / 16777216.0f);
      float x = 1.41421356237f * erfinvf(v);
      x = fminf(fmaxf(x, -2.0f), 2.0f);
      out[i] = copysignf(sqrtf(fabsf(x)), x);
    }
  }
}

__global__ void bump_counter_kernel(int64_t* counters, int which) {
  dz::pdl_enter(); counters[which] += 1; }

// ---- losses ------------------------------------------------------------------------------------

struct LossArgs {
  int kind, B, A, atoms, N, Ksel, Nt;  // N: #src quantiles (s_tm1), Ksel: selector samples, Nt: target samples
  const float* out0; const float* out1; const float* out2;       // head outputs of pass 0 / 1 / 2 (see learner)
  const float* adv0; const float* val0; const float* adv1; const float* val1; const float* adv2; const float* val2;  // rainbow
  const int32_t* a; const float* r; const float* disc; const float* w; const float* taus0;
  float vmax, bound, kappa;
  float* dout; float* dadv; float* dval;      // gradients wrt pass-0 head outputs
  float* per_example; float* priorities; float* loss_terms;  // loss_terms[b] = w_b * loss_b
};

__device__ __forceinline__ float block_sum(float v, float* smem) {
  v = warp_sum(v);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) smem[threadIdx.x >> 5] = v;
  __syncthreads();
  float t = threadIdx.x < (blockDim.x >> 5) ? smem[threadIdx.x] : 0.f;
  if (threadIdx.x < 32) t = warp_sum(t);
  if (threadIdx.x == 0) smem[0] = t;
  __syncthreads();
  t = smem[0];
  __syncthreads();
  return t;
}
__device__ __forceinline__ float block_max(float v, float* smem) {
  v = warp_max(v);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) smem[threadIdx.x >> 5] = v;
  __syncthreads();
  float t = threadIdx.x < (blockDim.x >> 5) ? smem[threadIdx.x] : -INFINITY;
  if (threadIdx.x < 32) t = warp_max(t);
  if (threadIdx.x == 0) smem[0] = t;
  __syncthreads();
  t = smem[0];
  __syncthreads();
  return t;
}

// dqn / double_q / prioritized: rlax.q_learning / double_q_learning, clip_gradient, l2_loss.
__global__ void __launch_bounds__(64) loss_q_kernel(LossArgs L) {
  dz::pdl_enter();
  int b = blockIdx.x;
  if (threadIdx.x != 0) return;
  const float* q_tm1 = L.out0 + (long long)b * L.A;
  const float* q_sel = (L.kind == DZ_DQN ? L.out2 : L.out1) + (long long)b * L.A;
  const float* q_tgt = L.out2 + (long long)b * L.A;
  int best = 0;
  for (int a = 1; a < L.A; ++a)
    if (q_sel[a] > q_sel[best]) best = a;
  int at = L.a[b];
  float target = L.r[b] + L.disc[b] * q_tgt[best];
  float td = target - q_tm1[at];
  float w = L.w ? L.w[b] : 1.0f;
  float g = fminf(fmaxf(w * td / (float)L.B, -L.bound), L.bound);  // cotangent reaching clip_gradient
  for (int a = 0; a < L.A; ++a) L.dout[(long long)b * L.A + a] = (a == at) ? -g : 0.f;
  L.per_example[b] = td;
  if (L.priorities) L.priorities[b] = fabsf(td);                   // prioritized/agent.py:201
  L.loss_terms[b] = w * 0.5f * td * td;
}

// c51 / rainbow: categorical_[double_]q_learning with categorical_l2_project + cross entropy.
// One CTA (4 warps) per example.  Softmaxes run one warp per (pass, action) with shuffle reductions, so the
// whole kernel has five block barriers.
__device__ __forceinline__ float warp_sum_all(float v) { return warp_sum(v); }

__global__ void __launch_bounds__(128) loss_categorical_kernel(LossArgs L) {
  dz::pdl_enter();
  extern __shared__ float sm[];
  const int b = blockIdx.x, K = L.atoms, A = L.A, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  float* cm_sel = sm;            // [K] mean over actions of the selector-pass advantages (rainbow)
  float* cm_tgt = cm_sel + K;    // [K] same for the target pass
  float* cm_tm1 = cm_tgt + K;    // [K] same for the online(s_tm1) pass
  float* p_tgt = cm_tm1 + K;     // [K]
  float* proj = p_tgt + K;       // [K]
  float* p_tm1 = proj + K;       // [K] softmax(logits_tm1[a_tm1])
  float* qsel = p_tm1 + K;       // [A]
  float* scal = qsel + A;        // [4]: loss, sum(proj)
  const bool rb = L.kind == DZ_RAINBOW;
  auto support = [&](int i) { return (float)((double)(-L.vmax) + (double)i * (2.0 * (double)L.vmax / (double)(K - 1))); };

  // 0. dueling column means (networks.py:251: mean over the action axis)
  if (rb) {
    for (int k = tid; k < K; k += blockDim.x) {
      float m1 = 0.f, m2 = 0.f, m0 = 0.f;
      for (int a = 0; a < A; ++a) {
        m1 += L.adv1[((long long)b * A + a) * K + k];
        m2 += L.adv2[((long long)b * A + a) * K + k];
        m0 += L.adv0[((long long)b * A + a) * K + k];
      }
      cm_sel[k] = m1 / (float)A; cm_tgt[k] = m2 / (float)A; cm_tm1[k] = m0 / (float)A;
    }
  }
  __syncthreads();
  // logit k of (pass, action): pass 0 = online(s_tm1), 1 = selector, 2 = target
  auto logit_of = [&](int pass, int a, int k) -> float {
    if (rb) {
      const float* adv = pass == 0 ? L.adv0 : (pass == 1 ? L.adv1 : L.adv2);
      const float* val = pass == 0 ? L.val0 : (pass == 1 ? L.val1 : L.val2);
      const float* cm = pass == 0 ? cm_tm1 : (pass == 1 ? cm_sel : cm_tgt);
      return val[(long long)b * K + k] + adv[((long long)b * A + a) * K + k] - cm[k];
    }
    const float* out = pass == 0 ? L.out0 : L.out2;   // c51 selects with the target network
    return out[((long long)b * A + a) * K + k];
  };
  // warp-level softmax of (pass, a): returns this lane's max/denominator; optionally writes probabilities
  auto warp_softmax = [&](int pass, int a, float* probs, float& mx, float& den) {
    float m = -INFINITY;
    for (int k = lane; k < K; k += 32) m = fmaxf(m, logit_of(pass, a, k));
    mx = warp_max(m);
    float s = 0.f;
    for (int k = lane; k < K; k += 32) s += expf(logit_of(pass, a, k) - mx);
    den = warp_sum(s);
    if (probs)
      for (int k = lane; k < K; k += 32) probs[k] = expf(logit_of(pass, a, k) - mx) / den;
  };

  // 1. selector q-values, one warp per action
  for (int a = warp; a < A; a += 4) {
    float mx, den;
    warp_softmax(rb ? 1 : 2, a, nullptr, mx, den);
    float s = 0.f;
    for (int k = lane; k < K; k += 32) s += (expf(logit_of(rb ? 1 : 2, a, k) - mx) / den) * support(k);
    s = warp_sum(s);
    if (lane == 0) qsel[a] = s;
  }
  __syncthreads();
  int best = 0;
  for (int a = 1; a < A; ++a)
    if (qsel[a] > qsel[best]) best = a;
  const int at = L.a[b];
  // 2. target distribution (warp 0) and softmax of the taken action's online logits (warp 1)
  float mx_tm1 = 0.f, den_tm1 = 1.f;
  if (warp == 0) { float mx, den; warp_softmax(2, best, p_tgt, mx, den); }
  if (warp == 1) {
    warp_softmax(0, at, p_tm1, mx_tm1, den_tm1);
    if (lane == 0) { scal[2] = mx_tm1; scal[3] = den_tm1; }
  }
  __syncthreads();
  // 3. rlax.categorical_l2_project(r + discount*z, p, z)
  const float r = L.r[b], dsc = L.disc[b];
  const float zmin = support(0), zmax = support(K - 1);
  for (int i = tid; i < K; i += blockDim.x) {
    float zi = support(i);
    float dpos = (i + 1 < K ? support(i + 1) : support(0)) - zi;      // roll(z,-1) - z
    float dneg = zi - (i > 0 ? support(i - 1) : support(K - 1));      // z - roll(z,1)
    dpos = dpos > 0.f ? 1.0f / dpos : 0.f;
    dneg = dneg > 0.f ? 1.0f / dneg : 0.f;
    float acc = 0.f;
    for (int j = 0; j < K; ++j) {
      float zp = fminf(fmaxf(r + dsc * support(j), zmin), zmax);
      float delta = zp - zi;
      float dhat = delta >= 0.f ? delta * dpos : -(delta * dneg);
      acc += fminf(fmaxf(1.0f - dhat, 0.f), 1.0f) * p_tgt[j];
    }
    proj[i] = acc;
  }
  __syncthreads();
  // 4. cross entropy with log_softmax(logits_tm1[a_tm1]) (warp 0)
  if (warp == 0) {
    const float mx = scal[2], logden = logf(scal[3]);
    float ls = 0.f, ps = 0.f;
    for (int k = lane; k < K; k += 32) {
      ls += proj[k] * (logit_of(0, at, k) - mx - logden);
      ps += proj[k];
    }
    ls = warp_sum(ls); ps = warp_sum(ps);
    if (lane == 0) { scal[0] = -ls; scal[1] = ps; }
  }
  __syncthreads();
  const float loss = scal[0], psum = scal[1];
  const float w = L.w ? L.w[b] : 1.0f;
  const float cot = w / (float)L.B;
  // 5. gradient wrt the pass-0 head outputs
  if (rb) {
    for (int k = tid; k < K; k += blockDim.x) {
      float dl = cot * (p_tm1[k] * psum - proj[k]);
      L.dval[(long long)b * K + k] = dl;
      for (int a = 0; a < A; ++a)
        L.dadv[((long long)b * A + a) * K + k] = dl * ((a == at ? 1.0f : 0.0f) - 1.0f / (float)A);
    }
  } else {
    for (int i = tid; i < A * K; i += blockDim.x) {
      int a = i / K, k = i - a * K;
      L.dout[(long long)b * A * K + i] = (a == at) ? cot * (p_tm1[k] * psum - proj[k]) : 0.f;
    }
  }
  if (tid == 0) {
    L.per_example[b] = loss;
    if (L.priorities) L.priorities[b] = fminf(fmaxf(fabsf(loss), 0.f), 100.f);  // rainbow/agent.py:194
    L.loss_terms[b] = w * loss;
  }
}

// Same kernel with the example's head outputs staged in shared memory first (identical arithmetic, identical results):
// the default whenever 3 * A * atoms floats fit (they do for every standard configuration).
__global__ void __launch_bounds__(128) loss_categorical_staged_kernel(LossArgs L) {
  dz::pdl_enter();
  extern __shared__ float sm[];
  const int b = blockIdx.x, K = L.atoms, A = L.A, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  float* cm_sel = sm;            // [K] mean over actions of the selector-pass advantages (rainbow)
  float* cm_tgt = cm_sel + K;    // [K] same for the target pass
  float* cm_tm1 = cm_tgt + K;    // [K] same for the online(s_tm1) pass
  float* p_tgt = cm_tm1 + K;     // [K]
  float* proj = p_tgt + K;       // [K]
  float* p_tm1 = proj + K;       // [K] softmax(logits_tm1[a_tm1])
  float* qsel = p_tm1 + K;       // [A]
  float* scal = qsel + A;        // [4]: loss, sum(proj)
  float* zs = scal + 4;          // [K] support atoms
  float* st_adv = zs + K;        // [3][A*K] head outputs of this example for pass 0 / 1 / 2
  float* st_val = st_adv + 3 * A * K;   // [3][K] value-stream outputs (rainbow)
  const bool rb = L.kind == DZ_RAINBOW;
  // Everything this example's loss reads from the three head passes goes to shared memory in ONE round of coalesced,
  // independent loads; the phases below are then shared-memory arithmetic instead of ~10 dependent global round trips.
  {
    const float* __restrict__ a0 = (rb ? L.adv0 : L.out0) + (long long)b * A * K;
    const float* __restrict__ a1 = (rb ? L.adv1 : L.out2) + (long long)b * A * K;
    const float* __restrict__ a2 = (rb ? L.adv2 : L.out2) + (long long)b * A * K;
    for (int i = tid; i < A * K; i += blockDim.x) {
      const float x0 = a0[i], x1 = a1[i], x2 = a2[i];
      st_adv[i] = x0; st_adv[A * K + i] = x1; st_adv[2 * A * K + i] = x2;
    }
    if (rb) {
      const float* __restrict__ v0 = L.val0 + (long long)b * K;
      const float* __restrict__ v1 = L.val1 + (long long)b * K;
      const float* __restrict__ v2 = L.val2 + (long long)b * K;
      for (int i = tid; i < K; i += blockDim.x) {
        const float x0 = v0[i], x1 = v1[i], x2 = v2[i];
        st_val[i] = x0; st_val[K + i] = x1; st_val[2 * K + i] = x2;
      }
    }
    for (int i = tid; i < K; i += blockDim.x) zs[i] = (float)((double)(-L.vmax) + (double)i * (2.0 * (double)L.vmax / (double)(K - 1)));
  }
  __syncthreads();
  auto support = [&](int i) { return zs[i]; };

  // 0. dueling column means (networks.py:251: mean over the action axis)
  if (rb) {
    for (int k = tid; k < K; k += blockDim.x) {
      float m1 = 0.f, m2 = 0.f, m0 = 0.f;
      for (int a = 0; a < A; ++a) {
        m1 += st_adv[A * K + a * K + k];
        m2 += st_adv[2 * A * K + a * K + k];
        m0 += st_adv[a * K + k];
      }
      cm_sel[k] = m1 / (float)A; cm_tgt[k] = m2 / (float)A; cm_tm1[k] = m0 / (float)A;
    }
  }
  __syncthreads();
  // logit k of (pass, action): pass 0 = online(s_tm1), 1 = selector, 2 = target
  auto logit_of = [&](int pass, int a, int k) -> float {
    if (rb) {
      const float* cm = pass == 0 ? cm_tm1 : (pass == 1 ? cm_sel : cm_tgt);
      return st_val[pass * K + k] + st_adv[pass * A * K + a * K + k] - cm[k];
    }
    return st_adv[(pass == 0 ? 0 : 2) * A * K + a * K + k];   // c51 selects with the target network
  };
  // warp-level softmax of (pass, a): returns this lane's max/denominator; optionally writes probabilities
  auto warp_softmax = [&](int pass, int a, float* probs, float& mx, float& den) {
    float m = -INFINITY;
    for (int k = lane; k < K; k += 32) m = fmaxf(m, logit_of(pass, a, k));
    mx = warp_max(m);
    float s = 0.f;
    for (int k = lane; k < K; k += 32) s += expf(logit_of(pass, a, k) - mx);
    den = warp_sum(s);
    if (probs)
      for (int k = lane; k < K; k += 32) probs[k] = expf(logit_of(pass, a, k) - mx) / den;
  };

  // 1. selector q-values, one warp per action
  for (int a = warp; a < A; a += 4) {
    float mx, den;
    warp_softmax(rb ? 1 : 2, a, nullptr, mx, den);
    float s = 0.f;
    for (int k = lane; k < K; k += 32) s += (expf(logit_of(rb ? 1 : 2, a, k) - mx) / den) * support(k);
    s = warp_sum(s);
    if (lane == 0) qsel[a] = s;
  }
  __syncthreads();
  int best = 0;
  for (int a = 1; a < A; ++a)
    if (qsel[a] > qsel[best]) best = a;
  const int at = L.a[b];
  // 2. target distribution (warp 0) and softmax of the taken action's online logits (warp 1)
  float mx_tm1 = 0.f, den_tm1 = 1.f;
  if (warp == 0) { float mx, den; warp_softmax(2, best, p_tgt, mx, den); }
  if (warp == 1) {
    warp_softmax(0, at, p_tm1, mx_tm1, den_tm1);
    if (lane == 0) { scal[2] = mx_tm1; scal[3] = den_tm1; }
  }
  __syncthreads();
  // 3. rlax.categorical_l2_project(r + discount*z, p, z)
  const float r = L.r[b], dsc = L.disc[b];
  const float zmin = support(0), zmax = support(K - 1);
  for (int i = tid; i < K; i += blockDim.x) {
    float zi = support(i);
    float dpos = (i + 1 < K ? support(i + 1) : support(0)) - zi;      // roll(z,-1) - z
    float dneg = zi - (i > 0 ? support(i - 1) : support(K - 1));      // z - roll(z,1)
    dpos = dpos > 0.f ? 1.0f / dpos : 0.f;
    dneg = dneg > 0.f ? 1.0f / dneg : 0.f;
    float acc = 0.f;
    for (int j = 0; j < K; ++j) {
      float zp = fminf(fmaxf(r + dsc * support(j), zmin), zmax);
      float delta = zp - zi;
      float dhat = delta >= 0.f ? delta * dpos : -(delta * dneg);
      acc += fminf(fmaxf(1.0f - dhat, 0.f), 1.0f) * p_tgt[j];
    }
    proj[i] = acc;
  }
  __syncthreads();
  // 4. cross entropy with log_softmax(logits_tm1[a_tm1]) (warp 0)
  if (warp == 0) {
    const float mx = scal[2], logden = logf(scal[3]);
    float ls = 0.f, ps = 0.f;
    for (int k = lane; k < K; k += 32) {
      ls += proj[k] * (logit_of(0, at, k) - mx - logden);
      ps += proj[k];
    }
    ls = warp_sum(ls); ps = warp_sum(ps);
    if (lane == 0) { scal[0] = -ls; scal[1] = ps; }
  }
  __syncthreads();
  const float loss = scal[0], psum = scal[1];
  const float w = L.w ? L.w[b] : 1.0f;
  const float cot = w / (float)L.B;
  // 5. gradient wrt the pass-0 head outputs
  if (rb) {
    for (int k = tid; k < K; k += blockDim.x) {
      float dl = cot * (p_tm1[k] * psum - proj[k]);
      L.dval[(long long)b * K + k] = dl;
      for (int a = 0; a < A; ++a)
        L.dadv[((long long)b * A + a) * K + k] = dl * ((a == at ? 1.0f : 0.0f) - 1.0f / (float)A);
    }
  } else {
    for (int i = tid; i < A * K; i += blockDim.x) {
      int a = i / K, k = i - a * K;
      L.dout[(long long)b * A * K + i] = (a == at) ? cot * (p_tm1[k] * psum - proj[k]) : 0.f;
    }
  }
  if (tid == 0) {
    L.per_example[b] = loss;
    if (L.priorities) L.priorities[b] = fminf(fmaxf(fabsf(loss), 0.f), 100.f);  // rainbow/agent.py:194
    L.loss_terms[b] = w * loss;
  }
}

// qrdqn / iqn: rlax.quantile_q_learning with quantile_regression_loss (Huber kappa).
// Layouts: qrdqn out[b, q*A + a] (networks.py:308), iqn out[(b*N + n)*A + a] (networks.py:286-287).
__global__ void __launch_bounds__(256) loss_quantile_kernel(LossArgs L) {
  dz::pdl_enter();
  extern __shared__ float sm[];
  const int b = blockIdx.x, A = L.A, tid = threadIdx.x;
  const bool iqn = L.kind == DZ_IQN;
  const int N = L.N, Ks = L.Ksel, Nt = L.Nt;
  float* red = sm;            // [32]
  float* qsel = sm + 32;      // [A]
  float* tgt = qsel + A;      // [Nt]
  float* src = tgt + Nt;      // [N]
  float* tau = src + N;       // [N]
  // selector: mean over samples of the selector distribution (qrdqn: the target dist itself)
  const float* sel = iqn ? L.out1 + (long long)b * Ks * A : L.out2 + (long long)b * Nt * A;
  const int nsel = iqn ? Ks : Nt;
  for (int a = 0; a < A; ++a) {
    float s = 0.f;
    for (int j = tid; j < nsel; j += blockDim.x) s += sel[(long long)j * A + a];
    s = block_sum(s, red);
    if (tid == 0) qsel[a] = s / (float)nsel;
    __syncthreads();
  }
  int best = 0;
  for (int a = 1; a < A; ++a)
    if (qsel[a] > qsel[best]) best = a;
  const int at = L.a[b];
  const float r = L.r[b], dsc = L.disc[b];
  const float* dist_t = L.out2 + (long long)b * Nt * A;
  const float* dist_s = L.out0 + (long long)b * N * A;
  for (int j = tid; j < Nt; j += blockDim.x) tgt[j] = r + dsc * dist_t[(long long)j * A + best];
  for (int i = tid; i < N; i += blockDim.x) {
    src[i] = dist_s[(long long)i * A + at];
    tau[i] = iqn ? L.taus0[(long long)b * N + i] : ((float)i + 0.5f) / (float)N;  // qrdqn/run_atari.py:137
  }
  __syncthreads();
  const float kappa = L.kappa;
  const float w = L.w ? L.w[b] : 1.0f;
  const float cot = w / (float)L.B;
  float total = 0.f;
  for (int i = tid; i < N; i += blockDim.x) {
    float acc = 0.f, gacc = 0.f;
    for (int j = 0; j < Nt; ++j) {
      float delta = tgt[j] - src[i];
      float wt = fabsf(tau[i] - (delta < 0.f ? 1.0f : 0.0f));
      float ad = fabsf(delta);
      float l, dl;
      if (kappa > 0.f) {
        float q = fminf(ad, kappa);
        l = 0.5f * q * q + kappa * (ad - q);
        dl = fminf(fmaxf(delta, -kappa), kappa);
      } else {
        l = ad;
        dl = delta > 0.f ? 1.0f : (delta < 0.f ? -1.0f : 0.0f);
      }
      acc += wt * l;
      gacc += wt * dl;
    }
    total += acc / (float)Nt;
    float g = -cot * gacc / (float)Nt;  // d loss / d src_i  (delta = target - src)
    for (int a = 0; a < A; ++a) L.dout[((long long)b * N + i) * A + a] = (a == at) ? g : 0.f;
  }
  total = block_sum(total, red);
  if (tid == 0) {
    L.per_example[b] = total;
    L.loss_terms[b] = w * total;
  }
}

__global__ void loss_mean_kernel(const float* __restrict__ terms, int B, float* loss, float* max_seen, const float* priorities) {
  dz::pdl_enter();
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    float s = 0.f;
    for (int b = 0; b < B; ++b) s += terms[b];
    loss[0] = s / (float)B;
    if (max_seen && priorities) {
      float m = max_seen[0];
      for (int b = 0; b < B; ++b) m = fmaxf(m, priorities[b]);
      max_seen[0] = m;  // rainbow/agent.py:196-197
    }
  }
}

// q_values of one head pass (select_action): c51/rainbow expectation, qr/iqn mean, dqn identity.
// blockIdx.x = environment stream (batched acting); one block for the single-observation call.
__global__ void __launch_bounds__(128) q_values_kernel(int kind, int A, int atoms, int nq, float vmax, const float* out,
                                                       const float* adv, const float* val, float* q) {
  dz::pdl_enter();
  extern __shared__ float sm[];
  float* red = sm;
  float* logit = sm + 32;
  const int tid = threadIdx.x;
  {
    const long long e = blockIdx.x;
    const long long per_img = (kind == DZ_C51 || kind == DZ_RAINBOW) ? (long long)A * atoms
                              : ((kind == DZ_QRDQN || kind == DZ_IQN) ? (long long)nq * A : (long long)A);
    out += e * per_img; adv += e * per_img; if (val) val += e * atoms; q += e * A;
  }
  for (int a = 0; a < A; ++a) {
    float res;
    if (kind == DZ_C51 || kind == DZ_RAINBOW) {
      const int K = atoms;
      for (int k = tid; k < K; k += blockDim.x) {
        if (kind == DZ_RAINBOW) {
          float m = 0.f;
          for (int aa = 0; aa < A; ++aa) m += adv[aa * K + k];
          logit[k] = val[k] + adv[a * K + k] - m / (float)A;
        } else {
          logit[k] = out[a * K + k];
        }
      }
      __syncthreads();
      float m = -INFINITY;
      for (int k = tid; k < K; k += blockDim.x) m = fmaxf(m, logit[k]);
      m = block_max(m, red);
      float s = 0.f, e = 0.f;
      for (int k = tid; k < K; k += blockDim.x) {
        float p = expf(logit[k] - m);
        s += p;
        e += p * (float)((double)(-vmax) + (double)k * (2.0 * (double)vmax / (double)(K - 1)));
      }
      s = block_sum(s, red);
      e = block_sum(e, red);
      res = e / s;
    } else if (kind == DZ_QRDQN || kind == DZ_IQN) {
      float s = 0.f;
      for (int j = tid; j < nq; j += blockDim.x) s += out[(long long)j * A + a];
      res = block_sum(s, red) / (float)nq;
    } else {
      res = out[a];
    }
    if (tid == 0) q[a] = res;
    __syncthreads();
  }
}

// ---- optimizer ---------------------------------------------------------------------------------

// Sum of squares -> per-block partials; the last block to finish adds them in a fixed order
// (deterministic), publishes the global norm and bumps the optimizer step count.
// sumsq_only: norm_out[0] receives the SUM OF SQUARES of the range (the split global norm: the optimizer adds the
// conv-gradient partials written by the weight-gradient finish kernels and takes the root), user_norm is not written.
__global__ void __launch_bounds__(256) grad_norm_kernel(const float* __restrict__ g, long long n, float* partials,
                                                        unsigned int* ticket, float* norm_out, int64_t* counters, float* user_norm,
                                                        int sumsq_only) {
  dz::pdl_enter();
  __shared__ float s[32];
  __shared__ bool last;
  float acc = 0.f;
  const long long n4 = n >> 2;   // the blob is padded to a multiple of 4 floats
  const float4* g4 = reinterpret_cast<const float4*>(g);
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.x * blockDim.x) {
    float4 v = g4[i];
    acc = fmaf(v.x, v.x, acc); acc = fmaf(v.y, v.y, acc); acc = fmaf(v.z, v.z, acc); acc = fmaf(v.w, v.w, acc);
  }
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0) s[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.f;
    for (int i = 0; i < (blockDim.x >> 5); ++i) t += s[i];
    partials[blockIdx.x] = t;
    __threadfence();
    unsigned int done = atomicAdd(ticket, 1u);
    last = (done == gridDim.x - 1);
  }
  __syncthreads();
  if (last) {   // fixed-order tree over the per-block partials: deterministic whatever block finishes last
    __threadfence();
    float t = 0.f;
    for (unsigned int i = threadIdx.x; i < gridDim.x; i += blockDim.x) t += ((volatile float*)partials)[i];
    t = warp_sum(t);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) s[threadIdx.x >> 5] = t;
    __syncthreads();
    if (threadIdx.x == 0) {
      float tot = 0.f;
      for (int i = 0; i < (blockDim.x >> 5); ++i) tot += s[i];
      norm_out[0] = sumsq_only ? tot : sqrtf(tot);
      if (user_norm && !sumsq_only) user_norm[0] = norm_out[0];
      *ticket = 0;
      counters[0] += 1;  // optax adam `count` (also counts rmsprop steps)
    }
  }
}

struct OptArgs {
  int kind; float lr, eps, decay, b1, b2, max_norm;
  float* p; const float* g; float* m; float* v; long long n; const float* norm; const int64_t* counters;
  // split global norm (tcgen05 path): norm = sqrt(fc_sumsq[0] + sum of parts[0..nparts)), recomputed identically by every block
  const float* parts; int nparts; const float* fc_sumsq; float* norm_out; float* user_norm;
  int stages;   // optimizer_bulk_kernel: depth of the shared-memory ring
};

// Fixed-order block reduction of the split-norm partials: every block of every launch gets the same bits.
__device__ __forceinline__ float split_norm(const float* __restrict__ parts, int nparts, const float* __restrict__ fc_sumsq) {
  __shared__ float s_red[8];
  float t = 0.f;
  if (threadIdx.x < 256) {   // the first 256 threads reduce (blocks of 256 or 512 threads): one fixed order
    for (int i = threadIdx.x; i < nparts; i += 256) t += __ldcg(parts + i);
    t = warp_sum(t);
    if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = t;
  }
  __syncthreads();
  float tot = __ldcg(fc_sumsq);
#pragma unroll
  for (int i = 0; i < 8; ++i) tot += s_red[i];
  return sqrtf(tot);
}

__global__ void __launch_bounds__(256) norm_finalize_kernel(const float* parts, int nparts, const float* fc_sumsq, float* norm_out,
                                                            float* user_norm) {
  dz::pdl_enter();
  const float norm = split_norm(parts, nparts, fc_sumsq);
  if (threadIdx.x == 0) { norm_out[0] = norm; if (user_norm) user_norm[0] = norm; }
}

// One parameter.  optax.scale_by_adam divides the moments by (1 - b^t) per element; here the two
// reciprocals are formed once per thread and multiplied in (<= 1 ulp from the division), leaving one sqrt
// and one division per parameter instead of four IEEE-division sequences: the kernel was issue-bound.
template <int KIND>
__device__ __forceinline__ float opt_one(const OptArgs& o, float p, float g, float& m, float& v, bool clip, float norm,
                                         float inv_c1, float inv_c2) {
  if (clip) g = (g / norm) * o.max_norm;
  float upd;
  if (KIND == DZ_ADAM) {  // optax.scale_by_adam: eps outside the sqrt, bias-corrected moments
    float mu = o.b1 * m + (1.0f - o.b1) * g;
    float nu = o.b2 * v + (1.0f - o.b2) * g * g;
    // Moments of parameters whose gradient stays zero decay THROUGH the denormal range (0.9^t reaches 1e-38 after ~800
    // steps) and every warp that holds one takes the slow paths of the IEEE division / square root below: measured, the
    // optimizer launch went 42.7 -> 58.5 us between step 50 and step 4000 of a run.  A denormal moment cannot change a
    // parameter (|update| < 1e-38 / eps), so it is stored as zero.
    if (fabsf(mu) < 1.17549435e-38f) mu = 0.f;
    if (nu < 1.17549435e-38f) nu = 0.f;
    m = mu; v = nu;
    upd = (mu * inv_c1) / (sqrtf(nu * inv_c2) + o.eps);
  } else {                // optax.rmsprop(centered=True): eps inside the sqrt
    float mu = o.decay * m + (1.0f - o.decay) * g;
    float nu = o.decay * v + (1.0f - o.decay) * g * g;
    if (fabsf(mu) < 1.17549435e-38f) mu = 0.f;   // see the Adam branch: no denormal moments in memory
    if (nu < 1.17549435e-38f) nu = 0.f;
    m = mu; v = nu;
    upd = g * (1.0f / sqrtf(nu - mu * mu + o.eps));
  }
  return p - o.lr * upd;
}

// 7 floats of traffic per parameter (read p,g,m,v; write p,m,v), 16-byte accesses, 4 independent
// float4 quadruples per thread in flight.  Measured alternatives (rainbow, 52.7 us per launch incl. ~5 us of
// event overhead): ld.global.cs on the gradient and/or st.global.cs on the moments: no change (52.7 / 53.0 us);
// 4 quadruples per thread: 71 us (register pressure halves the resident threads); 4, 8, 12, 16 blocks per SM:
// 43.9 / 45.0 / 45.8 / 46.7 us.
template <int KIND>
__global__ void __launch_bounds__(256) optimizer_kernel(OptArgs o) {
  dz::pdl_enter();
  const long long n4 = o.n >> 2;
  float4* p4 = reinterpret_cast<float4*>(o.p);
  const float4* g4 = reinterpret_cast<const float4*>(o.g);
  float4* m4 = reinterpret_cast<float4*>(o.m);
  float4* v4 = reinterpret_cast<float4*>(o.v);
  constexpr int U = 2;
  const long long stride = (long long)gridDim.x * blockDim.x;
  const long long first = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  // the first batch of loads is issued BEFORE the norm is formed: the split-norm reduction (shared memory, a block
  // barrier, ~700 L2 reads per block) then hides behind the memory latency of the stream instead of preceding it
  float4 p[U], g[U], m[U], v[U];
#pragma unroll
  for (int u = 0; u < U; ++u) {
    long long i = first + u * stride;
    if (i < n4) { p[u] = p4[i]; g[u] = g4[i]; m[u] = m4[i]; v[u] = v4[i]; }
  }
  float norm;
  if (o.parts != nullptr) {
    norm = split_norm(o.parts, o.nparts, o.fc_sumsq);
    if (blockIdx.x == 0 && threadIdx.x == 0) { o.norm_out[0] = norm; if (o.user_norm) o.user_norm[0] = norm; }
  } else {
    norm = o.norm[0];
  }
  const bool clip = o.max_norm > 0.f && !(norm < o.max_norm);  // optax.clip_by_global_norm trigger
  float c1 = 1.f, c2 = 1.f;
  if (KIND == DZ_ADAM) {
    float t = (float)o.counters[0];
    c1 = 1.0f / (1.0f - powf(o.b1, t));
    c2 = 1.0f / (1.0f - powf(o.b2, t));
  }
  for (long long i0 = first; i0 < n4; i0 += stride * U) {
    if (i0 != first) {
#pragma unroll
      for (int u = 0; u < U; ++u) {
        long long i = i0 + u * stride;
        if (i < n4) { p[u] = p4[i]; g[u] = g4[i]; m[u] = m4[i]; v[u] = v4[i]; }
      }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      long long i = i0 + u * stride;
      if (i < n4) {
        p[u].x = opt_one<KIND>(o, p[u].x, g[u].x, m[u].x, v[u].x, clip, norm, c1, c2);
        p[u].y = opt_one<KIND>(o, p[u].y, g[u].y, m[u].y, v[u].y, clip, norm, c1, c2);
        p[u].z = opt_one<KIND>(o, p[u].z, g[u].z, m[u].z, v[u].z, clip, norm, c1, c2);
        p[u].w = opt_one<KIND>(o, p[u].w, g[u].w, m[u].w, v[u].w, clip, norm, c1, c2);
        p4[i] = p[u]; m4[i] = m[u]; v4[i] = v[u];
      }
    }
  }
}

// The same update as a bulk-copy (TMA 1-D) pipeline: the four streams of a 256-quadruple chunk land in shared memory by
// cp.async.bulk (one elected thread, mbarrier complete_tx), 256 threads update them in place, and p / m / v leave by
// cp.async.bulk stores.  Memory-level parallelism no longer depends on registers x resident warps: every CTA keeps
// `stages` - 1 chunks (16 KB each) of loads in flight while it computes, and the LSU sees shared-memory traffic only.
// Identical arithmetic (opt_one), identical results.
constexpr int kOptStagesMax = 8;
constexpr int kOptChunk = 256;                            // float4 per stream per stage = one per thread
constexpr int kOptStageBytes = 4 * kOptChunk * 16;        // p, g, m, v

__device__ __forceinline__ void opt_bulk_load(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(tc::smem_u32(dst)),
               "l"(__cvta_generic_to_global(src)), "r"(bytes), "r"(tc::smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void opt_bulk_store(void* dst, const void* src, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(__cvta_generic_to_global(dst)),
               "r"(tc::smem_u32(src)), "r"(bytes)
               : "memory");
}

template <int KIND, int V>   // V floats per thread and stage: 4 (256 threads) or 2 (512 threads, twice the warps per byte of shared memory)
__global__ void __launch_bounds__(kOptChunk * 4 / V, V == 2 ? 4 : 1) optimizer_bulk_kernel(OptArgs o) {
  extern __shared__ __align__(128) unsigned char opt_sm[];
  const int kOptStages = o.stages;
  uint64_t* full = reinterpret_cast<uint64_t*>(opt_sm + kOptStages * kOptStageBytes);
  const int tid = threadIdx.x;
  const long long n4 = o.n >> 2;
  const long long nchunks = (n4 + kOptChunk - 1) / kOptChunk;
  const long long mine = blockIdx.x < nchunks ? (nchunks - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;   // chunks of this CTA
  float4* p4 = reinterpret_cast<float4*>(o.p);
  const float4* g4 = reinterpret_cast<const float4*>(o.g);
  float4* m4 = reinterpret_cast<float4*>(o.m);
  float4* v4 = reinterpret_cast<float4*>(o.v);
  if (tid == 0) {
    for (int s = 0; s < kOptStages; ++s) tc::mbar_init(&full[s], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  dz::pdl_enter();
  auto issue = [&](long long it, int s) {   // thread 0: loads of this CTA's it-th chunk into stage s = it % stages
    const long long c = blockIdx.x + it * gridDim.x;
    const long long q0 = c * kOptChunk;
    const uint32_t bytes = (uint32_t)(min((long long)kOptChunk, n4 - q0) * 16);
    unsigned char* st = opt_sm + s * kOptStageBytes;
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(tc::smem_u32(&full[s])), "r"(4 * bytes) : "memory");
    opt_bulk_load(st, p4 + q0, bytes, &full[s]);
    opt_bulk_load(st + kOptChunk * 16, g4 + q0, bytes, &full[s]);
    opt_bulk_load(st + 2 * kOptChunk * 16, m4 + q0, bytes, &full[s]);
    opt_bulk_load(st + 3 * kOptChunk * 16, v4 + q0, bytes, &full[s]);
  };
  // the first loads are issued BEFORE the norm is formed (see optimizer_kernel)
  if (tid == 0)
    for (long long it = 0; it < mine && it < kOptStages; ++it) issue(it, (int)it);
  float norm;
  if (o.parts != nullptr) {
    norm = split_norm(o.parts, o.nparts, o.fc_sumsq);
    if (blockIdx.x == 0 && tid == 0) { o.norm_out[0] = norm; if (o.user_norm) o.user_norm[0] = norm; }
  } else {
    norm = o.norm[0];
  }
  const bool clip = o.max_norm > 0.f && !(norm < o.max_norm);  // optax.clip_by_global_norm trigger
  float c1 = 1.f, c2 = 1.f;
  if (KIND == DZ_ADAM) {
    float t = (float)o.counters[0];
    c1 = 1.0f / (1.0f - powf(o.b1, t));
    c2 = 1.0f / (1.0f - powf(o.b2, t));
  }
  int s = 0;
  uint32_t phase = 0;
  for (long long it = 0; it < mine; ++it) {
    const long long q0 = (blockIdx.x + it * gridDim.x) * (long long)kOptChunk;
    const int valid = (int)min((long long)kOptChunk, n4 - q0);
    float4* sp = reinterpret_cast<float4*>(opt_sm + s * kOptStageBytes);
    float4* sg = sp + kOptChunk;
    float4* smm = sp + 2 * kOptChunk;
    float4* sv = sp + 3 * kOptChunk;
    if (tid == 0 && it > 0) {   // refill the stage of iteration it - 1 as soon as its stores have finished READING it
      const long long next = it - 1 + kOptStages;
      if (next < mine) {
        asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
        issue(next, s == 0 ? kOptStages - 1 : s - 1);
      }
    }
    tc::mbar_wait(&full[s], phase);
    if (V == 4) {
      if (tid < valid) {
        float4 p = sp[tid], g = sg[tid], m = smm[tid], v = sv[tid];
        p.x = opt_one<KIND>(o, p.x, g.x, m.x, v.x, clip, norm, c1, c2);
        p.y = opt_one<KIND>(o, p.y, g.y, m.y, v.y, clip, norm, c1, c2);
        p.z = opt_one<KIND>(o, p.z, g.z, m.z, v.z, clip, norm, c1, c2);
        p.w = opt_one<KIND>(o, p.w, g.w, m.w, v.w, clip, norm, c1, c2);
        sp[tid] = p; smm[tid] = m; sv[tid] = v;
      }
    } else {
      if (tid < 2 * valid) {
        float2 p = reinterpret_cast<float2*>(sp)[tid], g = reinterpret_cast<float2*>(sg)[tid];
        float2 m = reinterpret_cast<float2*>(smm)[tid], v = reinterpret_cast<float2*>(sv)[tid];
        p.x = opt_one<KIND>(o, p.x, g.x, m.x, v.x, clip, norm, c1, c2);
        p.y = opt_one<KIND>(o, p.y, g.y, m.y, v.y, clip, norm, c1, c2);
        reinterpret_cast<float2*>(sp)[tid] = p; reinterpret_cast<float2*>(smm)[tid] = m; reinterpret_cast<float2*>(sv)[tid] = v;
      }
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic-proxy writes -> visible to the bulk stores
    __syncthreads();
    if (tid == 0) {
      const uint32_t bytes = (uint32_t)valid * 16;
      opt_bulk_store(p4 + q0, sp, bytes);
      opt_bulk_store(m4 + q0, smm, bytes);
      opt_bulk_store(v4 + q0, sv, bytes);
      asm volatile("cp.async.bulk.commit_group;" ::: "memory");
    }
    if (++s == kOptStages) { s = 0; phase ^= 1u; }
  }
  if (tid == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");   // stores complete before the grid does
}

// epsilon-greedy over q[E][A] (dqn/agent.py:121-127): first maximum wins, as np.argmax / jnp.argmax.
__global__ void act_select_kernel(const float* __restrict__ q, int A, int E, const float* __restrict__ explore, float eps,
                                  int32_t* __restrict__ actions) {
  dz::pdl_enter();
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= E) return;
  int best = 0;
  float bq = q[(long long)e * A];
  for (int a = 1; a < A; ++a) {
    const float v = q[(long long)e * A + a];
    if (v > bq) { bq = v; best = a; }
  }
  if (explore != nullptr && explore[e] < eps) best = min((int)(explore[E + e] * (float)A), A - 1);
  actions[e] = best;
}

__global__ void make_row_table_kernel(const uint8_t* base, long long stride, int n, const uint8_t** table) {
  dz::pdl_enter();
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) table[i] = base + (long long)i * stride;
}

}  // namespace

// ------------------------------------------------------------------------------------------------
// The learner object
// ------------------------------------------------------------------------------------------------

struct dz_learner {
  dz_learner_config cfg;
  dz_learner_buffers buf;
  Layout lay;
  Dims d;
  int B;           // train batch
  int n_head[3];   // rows per image in the head stage for pass 0/1/2 (IQN: tau samples; others 1)
  // workspace (floats unless noted)
  float *act1[3], *act2[3], *act3[3];
  float *h1[3][2], *out[3], *outv[3];      // rainbow: h1[p][0]=adv stream, [1]=val stream; out=adv, outv=val
  float *cosf[3], *hi[3], *E0;             // iqn
  float* nn_partial;                        // split-K partials for the M=batch FC layers and heads
  float* conv_partial;                      // split-K partials for conv2/conv3 forward
  float* conv1_partial;                     // split-K partials for conv1 forward (conv1_splits > 1)
  int conv1_splits;
  float* nt_partial;                        // split partials of the input-gradient (NT) GEMMs
  float *dout, *doutv, *dh1[2], *dact3, *dtmp[2], *dcol, *dact2, *dact1, *dhi;
  float* tn_partial[4];                     // conv1/2/3 wgrad partials, [3] = iqn head/embed partial
  float *loss_terms, *scalars;              // scalars: [0]=norm, [1]=shared-bias scratch.., [8..]=norm partials
  unsigned int* ticket;
  const uint8_t** rows_sample[2];           // row tables filled by the fused sampler
  const uint8_t** rows_act;                 // 1-entry table for q_values
  int32_t* s_a; float *s_r, *s_d, *s_w;     // sampler-produced batch scalars
  float *act_noise_zero;                    // zeros (acting without noise is never used; placeholder)
  float* q_scratch;
  int norm_blocks;
  int fc_splits, head_splits, conv_splits, nt_splits;
  // packed-operand tcgen05 path of the IQN 3136->512 layer (dz_tcp.cuh): hi/lo tile images + split partials
  bool pk_on;
  struct PkImg { float* hi; float* lo; int rows_pad, red_pad; };
  PkImg pk_act[3], pk_wT[2], pk_w, pk_actT, pk_dh1T, pk_dh1, pk_cos[3], pk_weT[2], pk_dET, pk_cosT;
  bool pk_embed_bwd;
  int pk_embed_wgrad_splits;
  float *pk_fwd_partial, *pk_wgrad_partial;
  int pk_fwd_splits, pk_wgrad_splits;
  // second stream for work that is off the critical path of the backward pass (weight gradients, priority
  // write-back, noise generation); under stream capture it becomes a parallel branch of the CUDA graph
  cudaStream_t side;
  cudaEvent_t ev_fork, ev_join;
  bool side_dirty;
  // third branch: the FC part of the split gradient norm and the conv2 weight gradient run beside the first side stream
  cudaStream_t side2;
  cudaEvent_t ev_fork2, ev_join2;
  bool side2_dirty;
  float* norm_parts;                        // split-norm slots written by the conv weight-gradient finish kernels
  // TMA-fed tcgen05 path of the batch-sized step (dz_umma_net.cu): torso + 3136 -> 512 layer(s), forward and input gradients
  UmNet* um;
  char* um_ws;
  int um_npass, um_set[3];
};

namespace {

constexpr int kNormBlocks = 592;

// The packed-operand tcgen05 kernels carry IQN's 3136->512 layer whenever every network apply has >= 1024 rows
// (DZ_PK_IQN=0 falls back to the fp32-FMA kernels, for A/B timing).
bool g_pk_iqn = true;
int g_fc_splits = 0;      // DZ_FC_SPLITS override
int g_conv1_splits = 1;   // DZ_CONV1_SPLITS: split-K of the conv1 forward GEMM (K = 256).  Measured: rainbow (3 applies,
                          // 600 tiles) 336 / 344 / 341 us per step for 1 / 2 / 3 splits, dqn (2 applies) 217 / 213 / 217 us:
                          // the extra finish launch eats the gain, so the default stays 1.
void read_env();

// Split count for a one-CTA-per-SM kernel: minimise (waves of 148 CTAs) x (k-blocks per split).
int pick_splits(int64_t tiles, int nkb, int max_splits) {
  int best = 1;
  int64_t best_cost = -1;
  for (int s = 1; s <= max_splits; ++s) {
    int64_t cost = ceil_div(tiles * s, 148) * (ceil_div(nkb, s) + 6);   // +6: pipeline fill/drain per CTA
    if (best_cost < 0 || cost < best_cost) { best_cost = cost; best = s; }
  }
  return best;
}

// DZ_UMMA=0 keeps every contraction on the fp32-FMA kernels (A/B timing, geometries the tcgen05 path does not cover).
bool g_umma = true;
int64_t noise_stride(const dz_learner_config& c, const Dims& d);
struct NoiseVecs;

UmNetDesc make_um_desc(const dz_learner* l);

int64_t carve(dz_learner* l, char* base) {
  const dz_learner_config& c = l->cfg;
  const Dims& d = l->d;
  const int B = c.batch;
  Bump w{base};
  const bool rb = c.kind == DZ_RAINBOW, iqn = c.kind == DZ_IQN;
  int nh[3] = {1, 1, 1};
  if (iqn) { nh[0] = c.tau_samples_s_tm1; nh[1] = c.tau_samples_policy; nh[2] = c.tau_samples_s_t; }
  for (int p = 0; p < 3; ++p) l->n_head[p] = nh[p];
  for (int p = 0; p < 3; ++p) {
    l->act1[p] = w.take<float>((int64_t)B * d.h1 * d.w1 * 32);
    l->act2[p] = w.take<float>((int64_t)B * d.h2 * d.w2 * 64);
    l->act3[p] = w.take<float>((int64_t)B * d.feat);
    int64_t rows = (int64_t)B * nh[p];
    l->h1[p][0] = w.take<float>(rows * 512);
    l->h1[p][1] = rb ? w.take<float>(rows * 512) : nullptr;
    l->out[p] = w.take<float>(rows * d.out);
    l->outv[p] = rb ? w.take<float>((int64_t)B * c.num_atoms) : nullptr;
    l->cosf[p] = iqn ? w.take<float>(rows * c.latent_dim) : nullptr;
    l->hi[p] = iqn ? w.take<float>(rows * d.feat) : nullptr;
  }
  l->E0 = iqn ? w.take<float>((int64_t)B * nh[0] * d.feat) : nullptr;
  l->fc_splits = g_fc_splits > 0 ? std::min(g_fc_splits, 64) : 14; l->head_splits = 8; l->conv_splits = 4; l->nt_splits = 8;
  {
    int64_t head_n = std::max<int64_t>(d.out, c.num_atoms);
    int64_t fc = (int64_t)kMaxProblems * l->fc_splits * 2 * B * 512;
    int64_t hd = (int64_t)kMaxProblems * l->head_splits * 2 * B * head_n;
    l->nn_partial = w.take<float>(std::max(fc, hd));
    l->conv_partial = w.take<float>((int64_t)3 * l->conv_splits * B * d.h2 * d.w2 * 64);
    l->conv1_splits = std::max(1, std::min(g_conv1_splits, 4));
    l->conv1_partial = l->conv1_splits > 1 ? w.take<float>((int64_t)3 * l->conv1_splits * B * d.h1 * d.w1 * 32) : nullptr;
    l->nt_partial = w.take<float>((int64_t)2 * l->nt_splits * 2 * B * std::max<int64_t>(d.feat, 512));
  }
  int64_t rows0 = (int64_t)B * nh[0];
  l->dout = w.take<float>(rows0 * d.out);
  l->doutv = rb ? w.take<float>((int64_t)B * c.num_atoms) : nullptr;
  l->dh1[0] = w.take<float>(rows0 * 512);
  l->dh1[1] = rb ? w.take<float>(rows0 * 512) : nullptr;
  l->dact3 = w.take<float>((int64_t)B * d.feat);
  l->dtmp[0] = rb ? w.take<float>((int64_t)B * d.feat) : nullptr;
  l->dtmp[1] = rb ? w.take<float>((int64_t)B * d.feat) : nullptr;
  int64_t col2 = (int64_t)B * d.h2 * d.w2 * 512, col3 = (int64_t)B * d.h3 * d.w3 * 576;
  l->dcol = w.take<float>(col2 > col3 ? col2 : col3);
  l->dact2 = w.take<float>((int64_t)B * d.h2 * d.w2 * 64);
  l->dact1 = w.take<float>((int64_t)B * d.h1 * d.w1 * 32);
  l->dhi = iqn ? w.take<float>(rows0 * d.feat) : nullptr;
  l->tn_partial[0] = w.take<float>((int64_t)64 * 257 * 32);
  l->tn_partial[1] = w.take<float>((int64_t)32 * 513 * 64);
  l->tn_partial[2] = w.take<float>((int64_t)32 * 577 * 64);
  l->tn_partial[3] = iqn ? w.take<float>((int64_t)16 * (c.latent_dim + 1) * d.feat + 16 * 513 * 64) : nullptr;
  l->pk_on = false; l->pk_embed_bwd = false;
  if (iqn && g_pk_iqn && rows0 >= 1024 && (int64_t)B * nh[1] >= 1024 && (int64_t)B * nh[2] >= 1024 && d.feat % 16 == 0 &&
      c.latent_dim <= 128 && rows0 % 4 == 0 && ((int64_t)B * nh[1]) % 4 == 0 && ((int64_t)B * nh[2]) % 4 == 0) {
    l->pk_on = true;
    auto img = [&](dz_learner::PkImg& im, int64_t rows, int64_t red, int row_tile) {
      im.rows_pad = (int)(ceil_div(rows, row_tile) * row_tile);
      im.red_pad = (int)(ceil_div(red, kPkKB) * kPkKB);
      im.hi = w.take<float>(pk_image_floats(im.rows_pad, im.red_pad));
      im.lo = w.take<float>(pk_image_floats(im.rows_pad, im.red_pad));
    };
    int64_t tiles = 0;
    for (int p = 0; p < 3; ++p) { img(l->pk_act[p], (int64_t)B * nh[p], d.feat, 128); tiles += l->pk_act[p].rows_pad / 128 * 2; }
    img(l->pk_wT[0], 512, d.feat, 256);
    img(l->pk_wT[1], 512, d.feat, 256);
    img(l->pk_w, d.feat, 512, 256);
    img(l->pk_actT, d.feat + 1, rows0, 128);
    img(l->pk_dh1T, 512, rows0, 256);
    img(l->pk_dh1, rows0, 512, 128);
    for (int p = 0; p < 3; ++p) img(l->pk_cos[p], (int64_t)B * nh[p], c.latent_dim, 128);
    img(l->pk_weT[0], d.feat, c.latent_dim, 256);
    img(l->pk_weT[1], d.feat, c.latent_dim, 256);
    l->pk_embed_bwd = nh[0] == 64 && d.feat % 64 == 0;
    if (l->pk_embed_bwd) {
      img(l->pk_dET, d.feat, rows0, 128);
      img(l->pk_cosT, c.latent_dim + 1, rows0, 256);
      l->pk_embed_wgrad_splits = pick_splits(l->pk_dET.rows_pad / 128, l->pk_dET.red_pad / kPkKB, 8);
    }
    l->pk_fwd_splits = pick_splits(tiles, l->pk_act[0].red_pad / kPkKB, 6);
    l->pk_wgrad_splits = pick_splits((int64_t)l->pk_actT.rows_pad / 128 * 2, l->pk_actT.red_pad / kPkKB, 8);
    int64_t fwd_rows = (int64_t)B * (nh[0] + nh[1] + nh[2]);
    l->pk_fwd_partial = w.take<float>((int64_t)l->pk_fwd_splits * fwd_rows * 512);
    l->pk_wgrad_partial = w.take<float>((int64_t)l->pk_wgrad_splits * (d.feat + 1) * 512);
  }
  l->loss_terms = w.take<float>(B);
  l->scalars = w.take<float>(8 + kNormBlocks + d.out + 64);
  l->ticket = w.take<unsigned int>(4);
  l->rows_sample[0] = w.take<const uint8_t*>(B);
  l->rows_sample[1] = w.take<const uint8_t*>(B);
  l->rows_act = w.take<const uint8_t*>(B > 4 ? B : 4);
  l->s_a = w.take<int32_t>(B);
  l->s_r = w.take<float>(B);
  l->s_d = w.take<float>(B);
  l->s_w = w.take<float>(B);
  l->q_scratch = w.take<float>(64);
  l->norm_parts = w.take<float>(1024);
  l->um_ws = nullptr;
  if (g_umma) {
    UmNetDesc ud = make_um_desc(l);
    if (um_net_supported(ud)) {
      int64_t bytes = um_net_workspace_bytes(ud);
      l->um_ws = w.take<char>(bytes);
      if (!base) l->um_ws = reinterpret_cast<char*>(1);   // size query: "enabled" marker only
    }
  }
  return w.used;
}

// Noise layout of ONE apply: adv1_in[feat] adv1_out[512] adv2_in[512] adv2_out[A*atoms] val1_in[feat]
// val1_out[512] val2_in[512] val2_out[atoms]; every vector starts on a 4-float boundary.
inline int64_t pad4(int64_t n) { return (n + 3) / 4 * 4; }
int64_t noise_stride(const dz_learner_config& c, const Dims& d) {
  return 2 * (pad4(d.feat) + 512 + 512) + pad4((int64_t)c.num_actions * c.num_atoms) + pad4(c.num_atoms);
}
struct NoiseVecs { const float *a1i, *a1o, *a2i, *a2o, *v1i, *v1o, *v2i, *v2o; };
NoiseVecs noise_of(const dz_learner_config& c, const Dims& d, const float* base, int apply) {
  const float* p = base + (int64_t)apply * noise_stride(c, d);
  NoiseVecs n;
  n.a1i = p; p += pad4(d.feat); n.a1o = p; p += 512; n.a2i = p; p += 512; n.a2o = p; p += pad4((int64_t)c.num_actions * c.num_atoms);
  n.v1i = p; p += pad4(d.feat); n.v1o = p; p += 512; n.v2i = p; p += 512; n.v2o = p;
  return n;
}

UmNetDesc make_um_desc(const dz_learner* l) {
  const dz_learner_config& c = l->cfg;
  const Dims& d = l->d;
  const Layout& L = l->lay;
  UmNetDesc u;
  memset(&u, 0, sizeof(u));
  const bool needs_online_st = c.kind == DZ_DOUBLE_Q || c.kind == DZ_PRIORITIZED || c.kind == DZ_RAINBOW;
  u.B = c.batch; u.H = d.H; u.W = d.W;
  u.npass = needs_online_st ? 3 : 2;
  u.pass_target[0] = 0; u.pass_target[1] = needs_online_st ? 0 : 1; u.pass_target[2] = 1;
  u.online = l->buf.d_online; u.target = l->buf.d_target;
  const char* cw[3] = {"conv1/w", "conv2/w", "conv3/w"};
  const char* cb[3] = {"conv1/b", "conv2/b", "conv3/b"};
  for (int i = 0; i < 3; ++i) { u.off_conv_w[i] = L.off(cw[i]); u.off_conv_b[i] = L.off(cb[i]); }
  u.use_fc = c.kind != DZ_IQN;
  u.nstream = c.kind == DZ_RAINBOW ? 2 : 1;
  u.noisy = c.kind == DZ_RAINBOW ? 1 : 0;
  if (c.kind == DZ_RAINBOW) {
    const char* st[2] = {"adv", "val"};
    for (int s = 0; s < 2; ++s) {
      std::string pre = std::string(st[s]) + "1/";
      u.off_fc_w[s] = L.off(pre + "mu/w"); u.off_fc_b[s] = L.off(pre + "mu/b");
      u.off_fc_sw[s] = L.off(pre + "sigma/w"); u.off_fc_sb[s] = L.off(pre + "sigma/b");
    }
    static float origin[1];
    NoiseVecs nz = noise_of(c, d, origin, 0);
    u.noise_stride = noise_stride(c, d);
    u.noise_off_in[0] = nz.a1i - origin; u.noise_off_out[0] = nz.a1o - origin;
    u.noise_off_in[1] = nz.v1i - origin; u.noise_off_out[1] = nz.v1o - origin;
    for (int p = 0; p < 3; ++p) u.noise_apply[p] = p;
  } else if (u.use_fc) {
    u.off_fc_w[0] = L.off("fc1/w"); u.off_fc_b[0] = L.off("fc1/b");
  }
  return u;
}

GemmProblem zero_problem() {
  GemmProblem p;
  memset(&p, 0, sizeof(p));
  p.splits = 1;
  p.mul_div = 1;
  p.fd_per = make_fastdiv(1); p.fd_ow = make_fastdiv(1); p.fd_seg = make_fastdiv(1);
  return p;
}

void set_conv(GemmProblem& p, int mode, const void* A, int nimg, int H, int W, int Cin, int KH, int KW, int S) {
  p.a_mode = mode; p.A = A; p.H = H; p.W = W; p.Cin = Cin; p.KW = KW; p.S = S;
  p.OH = conv_out(H, KH, S); p.OW = conv_out(W, KW, S);
  p.seg = KW * Cin;
  p.fd_per = make_fastdiv(p.OH * p.OW); p.fd_ow = make_fastdiv(p.OW); p.fd_seg = make_fastdiv(p.seg);
  p.M = nimg * p.OH * p.OW;
  p.K = KH * KW * Cin;
}

template <typename KernelT>
int launch_batch(const char* tag, KernelT kernel, const GemmBatch& gb, dim3 grid, int threads, void* stream) {
  DZ_LAUNCH_NAMED(tag, kernel, grid, threads, 0, stream, gb);
  return DZ_OK;
}

#define DZ_TRY(expr) do { int _s = (expr); if (_s != DZ_OK) return _s; } while (0)


void read_env() {
  g_pk_iqn = !(getenv("DZ_PK_IQN") != nullptr && std::string(getenv("DZ_PK_IQN")) == "0");
  g_fc_splits = getenv("DZ_FC_SPLITS") ? atoi(getenv("DZ_FC_SPLITS")) : 0;
  g_conv1_splits = getenv("DZ_CONV1_SPLITS") ? atoi(getenv("DZ_CONV1_SPLITS")) : 1;
  g_umma = !(getenv("DZ_UMMA") != nullptr && std::string(getenv("DZ_UMMA")) == "0");
}

// ---- NN launch helpers (tile shapes chosen by M / N) -------------------------------------------

int run_nn(const char* tag, GemmBatch& gb, bool dual, void* stream) {
  int maxM = 0, maxN = 0, maxS = 1;
  for (int i = 0; i < gb.n; ++i) {
    maxM = gb.p[i].M > maxM ? gb.p[i].M : maxM;
    maxN = gb.p[i].N > maxN ? gb.p[i].N : maxN;
    maxS = gb.p[i].splits > maxS ? gb.p[i].splits : maxS;
  }
  if (maxM <= 32) {
    dim3 grid((unsigned)ceil_div(maxN, 64), (unsigned)(ceil_div(maxM, 32) * maxS), gb.n);
    if (dual) return launch_batch(tag, gemm_nn_kernel<32, 64, 16, 2, 4, true>, gb, grid, 256, stream);
    return launch_batch(tag, gemm_nn_kernel<32, 64, 16, 2, 4, false>, gb, grid, 256, stream);
  }
  if (maxN <= 32 && !dual) {
    dim3 grid(1, (unsigned)(ceil_div(maxM, 64) * maxS), gb.n);
    return launch_batch(tag, gemm_nn_kernel<64, 32, 16, 4, 4, false>, gb, grid, 128, stream);
  }
  dim3 grid((unsigned)ceil_div(maxN, 64), (unsigned)(ceil_div(maxM, 64) * maxS), gb.n);
  if (dual) return launch_batch(tag, gemm_nn_kernel<64, 64, 16, 4, 4, true>, gb, grid, 256, stream);
  return launch_batch(tag, gemm_nn_kernel<64, 64, 16, 4, 4, false>, gb, grid, 256, stream);
}

int run_tn(const char* tag, GemmBatch& gb, void* stream) {
  int maxK = 0, maxN = 0, maxS = 1;
  for (int i = 0; i < gb.n; ++i) {
    int kext = gb.p[i].K + ((gb.p[i].Cb || gb.p[i].Cb2) ? 1 : 0);
    maxK = kext > maxK ? kext : maxK;
    maxN = gb.p[i].N > maxN ? gb.p[i].N : maxN;
    maxS = gb.p[i].splits > maxS ? gb.p[i].splits : maxS;
  }
  if (maxN <= 32) {
    dim3 grid(1, (unsigned)(ceil_div(maxK, 64) * maxS), gb.n);
    return launch_batch(tag, gemm_tn_kernel<64, 32, 16, 4, 2>, gb, grid, 256, stream);
  }
  dim3 grid((unsigned)ceil_div(maxN, 64), (unsigned)(ceil_div(maxK, 64) * maxS), gb.n);
  return launch_batch(tag, gemm_tn_kernel<64, 64, 16, 4, 4>, gb, grid, 256, stream);
}

int run_nt(const char* tag, GemmBatch& gb, bool dual, void* stream) {
  int maxM = 0, maxK = 0, maxS = 1;
  for (int i = 0; i < gb.n; ++i) {
    maxM = gb.p[i].M > maxM ? gb.p[i].M : maxM;
    maxK = gb.p[i].K > maxK ? gb.p[i].K : maxK;
    maxS = gb.p[i].splits > maxS ? gb.p[i].splits : maxS;
  }
  if (maxM <= 32) {
    dim3 grid((unsigned)ceil_div(maxK, 64), (unsigned)(ceil_div(maxM, 32) * maxS), gb.n);
    if (dual) return launch_batch(tag, gemm_nt_kernel<32, 64, 16, 2, 4, true>, gb, grid, 256, stream);
    return launch_batch(tag, gemm_nt_kernel<32, 64, 16, 2, 4, false>, gb, grid, 256, stream);
  }
  dim3 grid((unsigned)ceil_div(maxK, 64), (unsigned)(ceil_div(maxM, 64) * maxS), gb.n);
  if (dual) return launch_batch(tag, gemm_nt_kernel<64, 64, 16, 4, 4, true>, gb, grid, 256, stream);
  return launch_batch(tag, gemm_nt_kernel<64, 64, 16, 4, 4, false>, gb, grid, 256, stream);
}

int finish_nn(const GemmBatch& gb, float* const* outs, bool dual, void* stream) {
  FinishNNBatch fb;
  fb.n = gb.n;
  long long mx = 0;
  for (int i = 0; i < gb.n; ++i) {
    const GemmProblem& p = gb.p[i];
    fb.f[i] = FinishNN{p.C, p.splits, p.split_stride, p.M, p.N, dual ? 1 : 0, p.bias, p.bias2, p.c_scale, p.relu, p.bias_shared, outs[i]};
    long long t = (long long)p.M * p.N;
    mx = t > mx ? t : mx;
  }
  dim3 grid((unsigned)std::min<long long>(ceil_div(mx, 256), 148 * 8), gb.n);   // grid-stride kernels
  DZ_LAUNCH(finish_nn_kernel, grid, 256, 0, stream, fb);
  return DZ_OK;
}

struct Pass {        // one network.apply
  const float* params;     // online or target blob
  const uint8_t* const* rows;  // image row table
  int set;                 // torso activation set index (0..2)
  int head;                // head pass index (0..2)
  int apply;               // noise apply index (rainbow)
};

// ---- forward -----------------------------------------------------------------------------------

struct TorsoJob { const float* params; const uint8_t* const* rows; int set; };

int forward_torso(dz_learner* l, const TorsoJob* jobs, int njobs, int nimg, void* stream) {
  const Dims& d = l->d;
  const Layout& L = l->lay;
  GemmBatch gb;
  gb.n = njobs;
  float* outs1[kMaxProblems];
  for (int i = 0; i < njobs; ++i) {   // conv1: uint8 rows gathered in place (K1 + K2 of SURVEY §2.1)
    GemmProblem p = zero_problem();
    set_conv(p, A_CONV_U8, jobs[i].rows, nimg, d.H, d.W, d.C, 8, 8, 4);
    p.B = jobs[i].params + L.off("conv1/w"); p.bias = jobs[i].params + L.off("conv1/b");
    p.N = 32; p.ldb = 32; p.ldc = 32; p.relu = 1; p.C = l->act1[jobs[i].set];
    outs1[i] = p.C;
    if (l->conv1_splits > 1 && nimg == l->B) {
      p.splits = l->conv1_splits; p.split_stride = (long long)p.M * 32;
      p.C = l->conv1_partial + (long long)i * p.splits * p.split_stride;
    }
    gb.p[i] = p;
  }
  DZ_TRY(run_nn("conv1_fwd", gb, false, stream));
  if (gb.p[0].splits > 1) DZ_TRY(finish_nn(gb, outs1, false, stream));
  // conv2 / conv3: few output tiles (41 / 25 per pass) -> split K four ways so the grid covers the 148 SMs;
  // finish_nn adds the bias and ReLU.
  for (int layer = 2; layer <= 3; ++layer) {
    float* outs[kMaxProblems];
    for (int i = 0; i < njobs; ++i) {
      GemmProblem p = zero_problem();
      if (layer == 2) {
        set_conv(p, A_CONV_F32, l->act1[jobs[i].set], nimg, d.h1, d.w1, 32, 4, 4, 2);
        p.B = jobs[i].params + L.off("conv2/w"); p.bias = jobs[i].params + L.off("conv2/b");
        outs[i] = l->act2[jobs[i].set];
      } else {
        set_conv(p, A_CONV_F32, l->act2[jobs[i].set], nimg, d.h2, d.w2, 64, 3, 3, 1);
        p.B = jobs[i].params + L.off("conv3/w"); p.bias = jobs[i].params + L.off("conv3/b");
        outs[i] = l->act3[jobs[i].set];
      }
      p.N = 64; p.ldb = 64; p.ldc = 64; p.relu = 1;
      p.splits = l->conv_splits; p.split_stride = (long long)p.M * 64;
      p.C = l->conv_partial + (long long)i * p.splits * p.split_stride;
      gb.p[i] = p;
    }
    DZ_TRY(run_nn(layer == 2 ? "conv2_fwd" : "conv3_fwd", gb, false, stream));
    DZ_TRY(finish_nn(gb, outs, false, stream));
  }
  return DZ_OK;
}

// Heads for the dqn / double_q / prioritized / c51 / qrdqn family.
int forward_heads_plain(dz_learner* l, const Pass* passes, int np, int nimg, void* stream, bool fc1_done = false) {
  const Dims& d = l->d;
  const Layout& L = l->lay;
  GemmBatch gb;
  gb.n = np;
  float* outs[kMaxProblems];
  const bool shared = l->cfg.kind == DZ_DOUBLE_Q || l->cfg.kind == DZ_PRIORITIZED;
  const int splits = nimg <= 32 ? l->fc_splits : 1;
  for (int i = 0; i < np && !fc1_done; ++i) {
    GemmProblem p = zero_problem();
    p.a_mode = A_PLAIN; p.A = l->act3[passes[i].set]; p.lda = d.feat; p.M = nimg; p.K = d.feat;
    p.B = passes[i].params + L.off("fc1/w"); p.N = 512; p.ldb = 512; p.ldc = 512;
    p.bias = passes[i].params + L.off("fc1/b"); p.relu = 1;
    outs[i] = l->h1[passes[i].head][0];
    if (splits > 1) {
      p.splits = splits; p.split_stride = (long long)nimg * 512;
      p.C = l->nn_partial + (long long)i * splits * p.split_stride;
    } else {
      p.C = outs[i];
    }
    gb.p[i] = p;
  }
  if (!fc1_done) {
    DZ_TRY(run_nn("fc1_fwd", gb, false, stream));
    if (splits > 1) DZ_TRY(finish_nn(gb, outs, false, stream));
  }
  for (int i = 0; i < np; ++i) {
    GemmProblem p = zero_problem();
    p.a_mode = A_PLAIN; p.A = l->h1[passes[i].head][0]; p.lda = 512; p.M = nimg; p.K = 512;
    p.B = passes[i].params + L.off("head/w"); p.N = d.out; p.ldb = d.out; p.ldc = d.out;
    p.bias = passes[i].params + L.off("head/b"); p.bias_shared = shared ? 1 : 0;
    outs[i] = l->out[passes[i].head];
    if (nimg <= 32) {
      p.splits = l->head_splits; p.split_stride = (long long)nimg * d.out;
      p.C = l->nn_partial + (long long)i * p.splits * p.split_stride;
    } else {
      p.C = outs[i];
    }
    gb.p[i] = p;
  }
  DZ_TRY(run_nn("head_fwd", gb, false, stream));
  if (nimg <= 32) DZ_TRY(finish_nn(gb, outs, false, stream));
  return DZ_OK;
}

// Rainbow: two noisy streams (networks.py:224-261, :137-178).
int forward_heads_rainbow(dz_learner* l, const Pass* passes, int np, int nimg, const float* noise, void* stream, bool fc1_done = false) {
  const Dims& d = l->d;
  const Layout& L = l->lay;
  const dz_learner_config& c = l->cfg;
  if (2 * np > kMaxProblems) return fail(DZ_EINVAL, "too many rainbow passes");
  GemmBatch gb;
  gb.n = 2 * np;
  float* outs[kMaxProblems];
  const int splits = nimg <= 32 ? l->fc_splits : 1;
  const char* st[2] = {"adv", "val"};
  for (int i = 0; i < np && !fc1_done; ++i) {
    NoiseVecs nz = noise_of(c, d, noise, passes[i].apply);
    for (int s = 0; s < 2; ++s) {
      std::string pre = std::string(st[s]) + "1/";
      GemmProblem p = zero_problem();
      p.a_mode = A_PLAIN; p.A = l->act3[passes[i].set]; p.lda = d.feat; p.M = nimg; p.K = d.feat;
      p.B = passes[i].params + L.off(pre + "mu/w"); p.B2 = passes[i].params + L.off(pre + "sigma/w");
      p.N = 512; p.ldb = 512; p.ldc = 512;
      p.bias = passes[i].params + L.off(pre + "mu/b"); p.bias2 = passes[i].params + L.off(pre + "sigma/b");
      p.a_scale = s == 0 ? nz.a1i : nz.v1i; p.c_scale = s == 0 ? nz.a1o : nz.v1o; p.relu = 1;
      int q = 2 * i + s;
      outs[q] = l->h1[passes[i].head][s];
      if (splits > 1) {
        p.splits = splits; p.split_stride = (long long)2 * nimg * 512;
        p.C = l->nn_partial + (long long)q * splits * p.split_stride;
      } else {
        p.C = outs[q];
      }
      gb.p[q] = p;
    }
  }
  if (!fc1_done) {
    DZ_TRY(run_nn("noisy1_fwd", gb, true, stream));
    if (splits > 1) DZ_TRY(finish_nn(gb, outs, true, stream));
  }
  for (int i = 0; i < np; ++i) {
    NoiseVecs nz = noise_of(c, d, noise, passes[i].apply);
    for (int s = 0; s < 2; ++s) {
      std::string pre = std::string(st[s]) + "2/";
      int n_out = s == 0 ? c.num_actions * c.num_atoms : c.num_atoms;
      GemmProblem p = zero_problem();
      p.a_mode = A_PLAIN; p.A = l->h1[passes[i].head][s]; p.lda = 512; p.M = nimg; p.K = 512;
      p.B = passes[i].params + L.off(pre + "mu/w"); p.B2 = passes[i].params + L.off(pre + "sigma/w");
      p.N = n_out; p.ldb = n_out; p.ldc = n_out;
      p.bias = nullptr; p.bias2 = passes[i].params + L.off(pre + "sigma/b");   // with_bias=False: mu has no bias
      p.a_scale = s == 0 ? nz.a2i : nz.v2i; p.c_scale = s == 0 ? nz.a2o : nz.v2o;
      int q = 2 * i + s;
      outs[q] = s == 0 ? l->out[passes[i].head] : l->outv[passes[i].head];
      if (nimg <= 32) {
        int64_t head_n = (int64_t)c.num_actions * c.num_atoms;
        p.splits = l->head_splits; p.split_stride = (long long)2 * nimg * n_out;
        p.C = l->nn_partial + (long long)q * l->head_splits * 2 * nimg * head_n;
      } else {
        p.C = outs[q];
      }
      gb.p[q] = p;
    }
  }
  DZ_TRY(run_nn("noisy2_fwd", gb, true, stream));
  if (nimg <= 32) DZ_TRY(finish_nn(gb, outs, true, stream));
  return DZ_OK;
}

// IQN embedding (latent -> 3136, ReLU, * state embedding) and 3136 -> 512 layer of the three network applies of
// one update on the packed-operand tcgen05 kernels: one pack launch (cosine features + every weight operand of
// this step), the embedding GEMM whose epilogue writes the hi/lo tile images of the next GEMMs directly (the fp32
// `hi` tensors are never materialised), the split fc1 GEMM, one finish (bias + ReLU).
int iqn_embed_fc1_forward_packed(dz_learner* l, const Pass* passes, const GemmBatch& fc1, bool keep_E0, void* stream) {
  const Dims& d = l->d;
  const Layout& L = l->lay;
  const dz_learner_config& c = l->cfg;
  PackBatch pb;
  memset(&pb, 0, sizeof(pb));
  const float* blob[2] = {nullptr, nullptr};   // distinct parameter blobs (online first)
  int widx[3];
  for (int i = 0; i < 3; ++i) {
    int k = 0;
    while (k < 2 && blob[k] && blob[k] != passes[i].params) ++k;
    if (k == 2) return fail(DZ_EINVAL, "iqn packed path expects at most two parameter blobs");
    blob[k] = passes[i].params; widx[i] = k;
    int hp = passes[i].head;
    const dz_learner::PkImg& im = l->pk_cos[hp];
    DZ_TRY(pk_add_job(pb, l->cosf[hp], c.latent_dim, 1, fc1.p[i].M, c.latent_dim, im.rows_pad, im.red_pad, -1, im.hi, im.lo));
  }
  for (int k = 0; k < 2; ++k) {
    if (!blob[k]) continue;
    DZ_TRY(pk_add_job(pb, blob[k] + L.off("embed/w"), d.feat, 0, d.feat, c.latent_dim, l->pk_weT[k].rows_pad, l->pk_weT[k].red_pad,
                      -1, l->pk_weT[k].hi, l->pk_weT[k].lo));
    DZ_TRY(pk_add_job(pb, blob[k] + L.off("fc1/w"), 512, 0, 512, d.feat, l->pk_wT[k].rows_pad, l->pk_wT[k].red_pad, -1,
                      l->pk_wT[k].hi, l->pk_wT[k].lo));
  }
  // backward-time operand that only depends on forward-time tensors: W (rows k, reduction n) for the input gradient
  DZ_TRY(pk_add_job(pb, l->buf.d_online + L.off("fc1/w"), 512, 1, d.feat, 512, l->pk_w.rows_pad, l->pk_w.red_pad, -1, l->pk_w.hi, l->pk_w.lo));
  DZ_TRY(launch_pack("iqn_pack_fwd", pb, stream));

  PkBatch eb;
  memset(&eb, 0, sizeof(eb));
  eb.n = 3;
  for (int i = 0; i < 3; ++i) {
    int hp = passes[i].head;
    PkProblem& p = eb.p[i];
    p.A = PkOperand{l->pk_cos[hp].hi, l->pk_cos[hp].lo, l->pk_cos[hp].rows_pad / 8};
    p.B = PkOperand{l->pk_weT[widx[i]].hi, l->pk_weT[widx[i]].lo, l->pk_weT[widx[i]].rows_pad / 8};
    p.MI = fc1.p[i].M; p.NJ = d.feat; p.nkb = l->pk_cos[hp].red_pad / kPkKB; p.splits = 1;
    p.bias_j = passes[i].params + L.off("embed/b");
    p.mul = l->act3[passes[i].set]; p.mul_div = l->n_head[hp]; p.mul_ld = d.feat;
    p.e0 = (keep_E0 && hp == 0) ? l->E0 : nullptr; p.e0_ld = d.feat;
    p.img_hi = l->pk_act[hp].hi; p.img_lo = l->pk_act[hp].lo; p.img_rg = l->pk_act[hp].rows_pad / 8;
    if (keep_E0 && hp == 0) { p.imgT_hi = l->pk_actT.hi; p.imgT_lo = l->pk_actT.lo; p.imgT_rg = l->pk_actT.rows_pad / 8; }
  }
  DZ_TRY(launch_pgemm("iqn_embed_fwd", eb, stream, 1));

  PkBatch kb;
  memset(&kb, 0, sizeof(kb));
  kb.n = 3;
  kb.run_kb = 2;     // forward: feeds the ReLU mask and the quantile targets -> fp32-FMA-chain accuracy
  GemmBatch fin = fc1;
  float* outs[kMaxProblems] = {nullptr};
  long long off = 0;
  for (int i = 0; i < 3; ++i) {
    int hp = passes[i].head;
    const dz_learner::PkImg& im = l->pk_act[hp];
    PkProblem& p = kb.p[i];
    p.A = PkOperand{im.hi, im.lo, im.rows_pad / 8};
    p.B = PkOperand{l->pk_wT[widx[i]].hi, l->pk_wT[widx[i]].lo, l->pk_wT[widx[i]].rows_pad / 8};
    p.MI = fc1.p[i].M; p.NJ = 512; p.nkb = im.red_pad / kPkKB;
    p.sc_i = 512; p.sc_j = 1; p.splits = l->pk_fwd_splits;
    p.split_stride = (long long)p.MI * 512;
    p.C = l->pk_fwd_partial + off;
    off += (long long)p.splits * p.split_stride;
    p.bias_j = fc1.p[i].bias; p.relu = 1;
    if (p.splits == 1) p.C = fc1.p[i].C;
    fin.p[i].C = p.C; fin.p[i].splits = p.splits; fin.p[i].split_stride = p.split_stride;
    outs[i] = fc1.p[i].C;
  }
  DZ_TRY(launch_pgemm("iqn_fc1_fwd", kb, stream));
  if (l->pk_fwd_splits > 1) DZ_TRY(finish_nn(fin, outs, false, stream));
  return DZ_OK;
}

// IQN (networks.py:264-292): cosine embedding -> linear -> relu -> * state embedding -> value head.
int forward_heads_iqn(dz_learner* l, const Pass* passes, int np, int nimg, const float* const* taus, bool keep_E0, void* stream) {
  const Dims& d = l->d;
  const Layout& L = l->lay;
  const dz_learner_config& c = l->cfg;
  GemmBatch gb;
  gb.n = np;
  for (int i = 0; i < np; ++i) {
    long long rows = (long long)nimg * l->n_head[passes[i].head];
    DZ_LAUNCH(iqn_cos_kernel, (unsigned)ceil_div(rows * c.latent_dim, 256), 256, 0, stream, taus[i], l->cosf[passes[i].head],
              rows, c.latent_dim);
  }
  const bool packed = l->pk_on && nimg == l->B && np == 3;
  if (!packed) {
    for (int i = 0; i < np; ++i) {
      int hp = passes[i].head;
      GemmProblem p = zero_problem();
      p.a_mode = A_PLAIN; p.A = l->cosf[hp]; p.lda = c.latent_dim; p.M = nimg * l->n_head[hp]; p.K = c.latent_dim;
      p.B = passes[i].params + L.off("embed/w"); p.N = d.feat; p.ldb = d.feat; p.ldc = d.feat;
      p.bias = passes[i].params + L.off("embed/b"); p.relu = 1;
      p.mul = l->act3[passes[i].set]; p.mul_div = l->n_head[hp];
      p.C = l->hi[hp]; p.C2 = (keep_E0 && hp == 0) ? l->E0 : nullptr;
      gb.p[i] = p;
    }
    DZ_TRY(run_nn("iqn_embed_fwd", gb, false, stream));
  }
  for (int i = 0; i < np; ++i) {
    int hp = passes[i].head;
    GemmProblem p = zero_problem();
    p.a_mode = A_PLAIN; p.A = l->hi[hp]; p.lda = d.feat; p.M = nimg * l->n_head[hp]; p.K = d.feat;
    p.B = passes[i].params + L.off("fc1/w"); p.N = 512; p.ldb = 512; p.ldc = 512;
    p.bias = passes[i].params + L.off("fc1/b"); p.relu = 1; p.C = l->h1[hp][0];
    gb.p[i] = p;
  }
  // M can be small when acting (1 x tau_samples_policy rows): same kernel family handles it
  if (packed) {
    DZ_TRY(iqn_embed_fc1_forward_packed(l, passes, gb, keep_E0, stream));
  } else {
    DZ_TRY(run_nn("iqn_fc1_fwd", gb, false, stream));
  }
  if ((long long)nimg * l->n_head[passes[0].head] >= 512 && d.out <= kSkinnyMaxN && np <= 3) {
    SkinnyHead h;
    memset(&h, 0, sizeof(h));
    h.n = np;
    int maxM = 0;
    for (int i = 0; i < np; ++i) {
      int hp = passes[i].head;
      h.A[i] = l->h1[hp][0]; h.W[i] = passes[i].params + L.off("head/w"); h.bias[i] = passes[i].params + L.off("head/b");
      h.out[i] = l->out[hp]; h.M[i] = nimg * l->n_head[hp];
      maxM = std::max(maxM, h.M[i]);
    }
    dim3 grid((unsigned)std::min<int64_t>(ceil_div(maxM, 8), 148 * 2), (unsigned)np);
    DZ_LAUNCH_NAMED("iqn_head_fwd", iqn_head_fwd_kernel, grid, 256, 0, stream, h, d.out);
    return DZ_OK;
  }
  for (int i = 0; i < np; ++i) {
    int hp = passes[i].head;
    GemmProblem p = zero_problem();
    p.a_mode = A_PLAIN; p.A = l->h1[hp][0]; p.lda = 512; p.M = nimg * l->n_head[hp]; p.K = 512;
    p.B = passes[i].params + L.off("head/w"); p.N = d.out; p.ldb = d.out; p.ldc = d.out;
    p.bias = passes[i].params + L.off("head/b"); p.C = l->out[hp];
    gb.p[i] = p;
  }
  DZ_TRY(run_nn("iqn_head_fwd", gb, false, stream));
  return DZ_OK;
}

// ---- backward ----------------------------------------------------------------------------------

FinishNT make_finish_nt(const GemmProblem* probs, int nsrc, const float* mask, float* out, bool dual, float* out_hi = nullptr,
                        float* out_lo = nullptr) {
  FinishNT f;
  memset(&f, 0, sizeof(f));
  f.nsrc = nsrc; f.splits = probs[0].splits; f.stride = probs[0].split_stride; f.M = probs[0].M; f.K = probs[0].K;
  f.dual = dual ? 1 : 0; f.mask = mask; f.out = out; f.out_hi = out_hi; f.out_lo = out_lo;
  for (int q = 0; q < nsrc; ++q) { f.partial[q] = probs[q].C; f.a_scale[q] = probs[q].a_scale; }
  return f;
}
int finish_nt_batch(const FinishNT* jobs, int njobs, void* stream) {
  FinishNTBatch fb;
  memset(&fb, 0, sizeof(fb));
  long long total = 0;
  for (int j = 0; j < njobs; ++j) { fb.f[j] = jobs[j]; total = std::max(total, (long long)jobs[j].M * jobs[j].K); }
  dim3 grid((unsigned)std::min<long long>(ceil_div(total, 256), 148 * 8), (unsigned)njobs);
  DZ_LAUNCH(finish_nt_kernel, grid, 256, 0, stream, fb);
  return DZ_OK;
}
int finish_nt(const GemmProblem* probs, int nsrc, const float* mask, float* out, bool dual, void* stream) {
  FinishNT f = make_finish_nt(probs, nsrc, mask, out, dual);
  return finish_nt_batch(&f, 1, stream);
}

// Returns the side stream after making it wait for everything enqueued on `stream` so far (or `stream`
// itself when there is no side stream).  join_side() makes `stream` wait for the side work again.
void* fork_side(dz_learner* l, void* stream) {
  if (!l->side) return stream;
  if (cudaEventRecord(l->ev_fork, (cudaStream_t)stream) != cudaSuccess) return stream;
  if (cudaStreamWaitEvent(l->side, l->ev_fork, 0) != cudaSuccess) return stream;
  l->side_dirty = true;
  return l->side;
}
int join_side(dz_learner* l, void* stream) {
  if (!l->side || !l->side_dirty) return DZ_OK;
  DZ_CUDA_OK(cudaEventRecord(l->ev_join, l->side));
  DZ_CUDA_OK(cudaStreamWaitEvent((cudaStream_t)stream, l->ev_join, 0));
  l->side_dirty = false;
  return DZ_OK;
}
// Second side stream: `from` is the stream whose enqueued work it must wait for (the main stream or the first side stream).
void* fork_side2(dz_learner* l, void* from, void* fallback) {
  if (!l->side2) return fallback;
  if (cudaEventRecord(l->ev_fork2, (cudaStream_t)from) != cudaSuccess) return fallback;
  if (cudaStreamWaitEvent(l->side2, l->ev_fork2, 0) != cudaSuccess) return fallback;
  l->side2_dirty = true;
  return l->side2;
}
int join_side2(dz_learner* l, void* stream) {
  if (!l->side2 || !l->side2_dirty) return DZ_OK;
  DZ_CUDA_OK(cudaEventRecord(l->ev_join2, l->side2));
  DZ_CUDA_OK(cudaStreamWaitEvent((cudaStream_t)stream, l->ev_join2, 0));
  l->side2_dirty = false;
  return DZ_OK;
}
bool split_norm_active(const dz_learner* l);

// Torso backward from dact3 (already masked by act3 > 0): conv3/conv2/conv1 weight+bias grads.
int backward_torso(dz_learner* l, const uint8_t* const* rows0, void* stream) {
  const Dims& d = l->d;
  const Layout& L = l->lay;
  const int B = l->B;
  float* G = l->buf.d_grads;
  const float* P = l->buf.d_online;
  FinishTNBatch fb;
  fb.n = 0;
  GemmBatch gb;
  if (l->um && l->cfg.kind == DZ_IQN) DZ_TRY(um_split_dact3(l->um, stream));   // dact3 came from the Hadamard kernel (fp32)
  // conv3 wgrad
  float* norm_parts = split_norm_active(l) ? l->norm_parts : nullptr;
  if (l->um) {   // conv3 weight gradient + its finish (partial sums, bias gradient, split-norm partials) on the side stream
    void* ws = fork_side(l, stream);
    DZ_TRY(um_wgrad_conv3(l->um, ws));
    DZ_TRY(um_wgrad_finish_layer(l->um, 3, G + L.off("conv3/w"), G + L.off("conv3/b"), norm_parts, ws));
  } else {
    GemmProblem p = zero_problem();
    set_conv(p, A_CONV_F32, l->act2[0], B, d.h2, d.w2, 64, 3, 3, 1);
    p.B = l->dact3; p.N = 64; p.ldb = 64; p.ldc = 64;
    p.Cb = G + L.off("conv3/b");
    int splits = (int)std::min<int64_t>(32, ceil_div(p.M, 64));
    p.splits = splits; p.split_stride = (long long)(p.K + 1) * 64; p.C = l->tn_partial[2];
    gb.n = 1; gb.p[0] = p;
    DZ_TRY(run_tn("conv3_wgrad", gb, fork_side(l, stream)));
    fb.f[fb.n++] = FinishTN{p.C, splits, p.split_stride, p.K, 64, G + L.off("conv3/w"), nullptr, p.Cb, nullptr, nullptr, nullptr};
  }
  // conv3 dgrad: dcol = dpre3 * W3^T ; col2im with ReLU mask of act2
  if (l->um) {
    DZ_TRY(um_backward_conv3(l->um, stream));
  } else {
    GemmProblem p = zero_problem();
    p.A = l->dact3; p.lda = 64; p.M = B * d.h3 * d.w3; p.N = 64; p.K = 576;
    p.B = P + L.off("conv3/w"); p.ldb = 64; p.C = l->dcol; p.ldc = 576;
    gb.n = 1; gb.p[0] = p;
    DZ_TRY(run_nt("conv3_dgrad", gb, false, stream));
    long long total = (long long)B * d.h2 * d.w2 * 64;
    DZ_LAUNCH(col2im_kernel, (unsigned)ceil_div(total, 256), 256, 0, stream, l->dcol, l->act2[0], l->dact2, B, d.h2, d.w2, 64, 3, 3, 1,
              d.h3, d.w3);
  }
  // conv2 wgrad
  if (l->um) {   // conv2: on the second side stream, beside conv3's (both fit next to the input-gradient kernels)
    void* ws = l->side2 ? fork_side2(l, stream, stream) : fork_side(l, stream);
    DZ_TRY(um_wgrad_conv2(l->um, ws));
    DZ_TRY(um_wgrad_finish_layer(l->um, 2, G + L.off("conv2/w"), G + L.off("conv2/b"), norm_parts, ws));
  } else {
    GemmProblem p = zero_problem();
    set_conv(p, A_CONV_F32, l->act1[0], B, d.h1, d.w1, 32, 4, 4, 2);
    p.B = l->dact2; p.N = 64; p.ldb = 64; p.ldc = 64;
    p.Cb = G + L.off("conv2/b");
    int splits = (int)std::min<int64_t>(32, ceil_div(p.M, 64));
    p.splits = splits; p.split_stride = (long long)(p.K + 1) * 64; p.C = l->tn_partial[1];
    gb.n = 1; gb.p[0] = p;
    DZ_TRY(run_tn("conv2_wgrad", gb, fork_side(l, stream)));
    fb.f[fb.n++] = FinishTN{p.C, splits, p.split_stride, p.K, 64, G + L.off("conv2/w"), nullptr, p.Cb, nullptr, nullptr, nullptr};
  }
  // conv2 dgrad
  if (l->um) {
    DZ_TRY(um_backward_conv2(l->um, stream));
  } else {
    GemmProblem p = zero_problem();
    p.A = l->dact2; p.lda = 64; p.M = B * d.h2 * d.w2; p.N = 64; p.K = 512;
    p.B = P + L.off("conv2/w"); p.ldb = 64; p.C = l->dcol; p.ldc = 512;
    gb.n = 1; gb.p[0] = p;
    DZ_TRY(run_nt("conv2_dgrad", gb, false, stream));
    long long total = (long long)B * d.h1 * d.w1 * 32;
    DZ_LAUNCH(col2im_kernel, (unsigned)ceil_div(total, 256), 256, 0, stream, l->dcol, l->act1[0], l->dact1, B, d.h1, d.w1, 32, 4, 4, 2,
              d.h2, d.w2);
  }
  // conv1 wgrad (A = uint8 rows in place)
  if (l->um) {
    void* ws = fork_side(l, stream);
    DZ_TRY(um_wgrad_conv1(l->um, rows0, ws));
    DZ_TRY(um_wgrad_finish_layer(l->um, 1, G + L.off("conv1/w"), G + L.off("conv1/b"), norm_parts, ws));
    DZ_TRY(join_side2(l, stream));
    return join_side(l, stream);
  } else {
    GemmProblem p = zero_problem();
    set_conv(p, A_CONV_U8, rows0, B, d.H, d.W, d.C, 8, 8, 4);
    p.B = l->dact1; p.N = 32; p.ldb = 32; p.ldc = 32;
    p.Cb = G + L.off("conv1/b");
    int splits = (int)std::min<int64_t>(64, ceil_div(p.M, 64));
    p.splits = splits; p.split_stride = (long long)(p.K + 1) * 32; p.C = l->tn_partial[0];
    gb.n = 1; gb.p[0] = p;
    DZ_TRY(run_tn("conv1_wgrad", gb, fork_side(l, stream)));
    fb.f[fb.n++] = FinishTN{p.C, splits, p.split_stride, p.K, 32, G + L.off("conv1/w"), nullptr, p.Cb, nullptr, nullptr, nullptr};
  }
  void* ws = l->side && l->side_dirty ? (void*)l->side : stream;   // after conv1_wgrad on the same (side) stream
  dim3 grid((unsigned)ceil_div(577 * 64, 256), fb.n);
  DZ_LAUNCH(finish_tn_kernel, grid, 256, 0, ws, fb);
  return join_side(l, stream);
}

int backward_plain(dz_learner* l, void* stream) {
  const Dims& d = l->d;
  const Layout& L = l->lay;
  const int B = l->B;
  float* G = l->buf.d_grads;
  const float* P = l->buf.d_online;
  const bool shared = l->cfg.kind == DZ_DOUBLE_Q || l->cfg.kind == DZ_PRIORITIZED;
  GemmBatch gb;
  gb.n = 1;
  {  // head wgrad
    GemmProblem p = zero_problem();
    p.a_mode = A_PLAIN; p.A = l->h1[0][0]; p.lda = 512; p.M = B; p.K = 512;
    p.B = l->dout; p.N = d.out; p.ldb = d.out; p.ldc = d.out;
    p.C = G + L.off("head/w"); p.Cb = shared ? l->scalars + 8 + kNormBlocks : G + L.off("head/b");
    gb.p[0] = p;
    DZ_TRY(run_tn("head_wgrad", gb, fork_side(l, stream)));
    if (shared) DZ_LAUNCH(sum_to_scalar_kernel, 1, 128, 0, (l->side && l->side_dirty ? (void*)l->side : stream), l->scalars + 8 + kNormBlocks, d.out, G + L.off("head/b"));
  }
  bool dh1_split_done = false;
  {  // dh1 = dout * Wh^T, masked by h1 > 0
    GemmProblem p = zero_problem();
    p.A = l->dout; p.lda = d.out; p.M = B; p.N = d.out; p.K = 512;
    p.B = P + L.off("head/w"); p.ldb = d.out; p.C = l->dh1[0]; p.ldc = 512; p.mask = l->h1[0][0];
    // Wide heads (c51: 306 outputs, qr-dqn: 1206): with one CTA column per 64 outputs of dh1 the reduction over the head
    // width is a serial chain (measured 24 / 65 us); split it and let the finish kernel apply the mask (and, on the tcgen05
    // path, write the tf32 hi/lo pair fc1_dgrad reads, which saves the separate split launch).
    const int splits = d.out > 64 ? (int)std::min<int64_t>(16, ceil_div(d.out, 96)) : 1;
    if (splits > 1) {
      p.splits = splits; p.split_stride = (long long)B * 512; p.C = l->nt_partial; p.mask = nullptr;
      gb.p[0] = p;
      DZ_TRY(run_nt("head_dgrad", gb, false, stream));
      FinishNT job = make_finish_nt(&gb.p[0], 1, l->h1[0][0], l->dh1[0], false, l->um ? um_dh1_hi(l->um, 0) : nullptr,
                                    l->um ? um_dh1_lo(l->um, 0) : nullptr);
      DZ_TRY(finish_nt_batch(&job, 1, stream));
      dh1_split_done = l->um != nullptr;
    } else {
      gb.p[0] = p;
      DZ_TRY(run_nt("head_dgrad", gb, false, stream));
    }
  }
  {  // fc1 wgrad
    GemmProblem p = zero_problem();
    p.a_mode = A_PLAIN; p.A = l->act3[0]; p.lda = d.feat; p.M = B; p.K = d.feat;
    p.B = l->dh1[0]; p.N = 512; p.ldb = 512; p.ldc = 512;
    p.C = G + L.off("fc1/w"); p.Cb = G + L.off("fc1/b");
    gb.p[0] = p;
    DZ_TRY(run_tn("fc1_wgrad", gb, fork_side(l, stream)));
  }
  if (l->um) {   // dact3 on the tcgen05 path: dh1 -> tf32 hi/lo, W streamed once through TMA, split partials + masked finish
    if (!dh1_split_done) DZ_TRY(um_split_dh1(l->um, stream));
    DZ_TRY(um_backward_fc(l->um, nullptr, stream));
  } else {  // dact3 = dh1 * Wf^T, masked by act3 > 0
    GemmProblem p = zero_problem();
    p.A = l->dh1[0]; p.lda = 512; p.M = B; p.N = 512; p.K = d.feat;
    p.B = P + L.off("fc1/w"); p.ldb = 512; p.ldc = d.feat;
    // weight-streaming GEMM with a 32-row output: split the reduction so ~400 CTAs keep HBM busy
    p.splits = l->nt_splits; p.split_stride = (long long)B * d.feat; p.C = l->nt_partial;
    gb.p[0] = p;
    DZ_TRY(run_nt("fc1_dgrad", gb, false, stream));
    DZ_TRY(finish_nt(gb.p, 1, l->act3[0], l->dact3, false, stream));
  }
  return DZ_OK;
}

int backward_rainbow(dz_learner* l, const float* noise, void* stream) {
  const Dims& d = l->d;
  const Layout& L = l->lay;
  const dz_learner_config& c = l->cfg;
  const int B = l->B;
  float* G = l->buf.d_grads;
  const float* P = l->buf.d_online;
  NoiseVecs nz = noise_of(c, d, noise, 0);
  const char* st[2] = {"adv", "val"};
  GemmBatch gb;
  gb.n = 2;
  for (int s = 0; s < 2; ++s) {  // second noisy layer weight grads
    std::string pre = std::string(st[s]) + "2/";
    int n_out = s == 0 ? c.num_actions * c.num_atoms : c.num_atoms;
    GemmProblem p = zero_problem();
    p.a_mode = A_PLAIN; p.A = l->h1[0][s]; p.lda = 512; p.M = B; p.K = 512;
    p.B = s == 0 ? l->dout : l->doutv; p.N = n_out; p.ldb = n_out; p.ldc = n_out;
    p.C = G + L.off(pre + "mu/w"); p.C2 = G + L.off(pre + "sigma/w"); p.Cb = nullptr; p.Cb2 = G + L.off(pre + "sigma/b");
    p.a_scale = s == 0 ? nz.a2i : nz.v2i; p.c_scale = s == 0 ? nz.a2o : nz.v2o;
    gb.p[s] = p;
  }
  DZ_TRY(run_tn("noisy2_wgrad", gb, fork_side(l, stream)));
  for (int s = 0; s < 2; ++s) {  // dh1_s
    std::string pre = std::string(st[s]) + "2/";
    int n_out = s == 0 ? c.num_actions * c.num_atoms : c.num_atoms;
    GemmProblem p = zero_problem();
    p.A = s == 0 ? l->dout : l->doutv; p.lda = n_out; p.M = B; p.N = n_out; p.K = 512;
    p.B = P + L.off(pre + "mu/w"); p.B2 = P + L.off(pre + "sigma/w"); p.ldb = n_out;
    p.a_scale = s == 0 ? nz.a2i : nz.v2i; p.c_scale = s == 0 ? nz.a2o : nz.v2o;
    p.ldc = 512;
    p.splits = 4; p.split_stride = (long long)2 * B * 512;
    p.C = l->nt_partial + (long long)s * 4 * p.split_stride;
    gb.p[s] = p;
  }
  DZ_TRY(run_nt("noisy2_dgrad", gb, true, stream));
  {   // both streams' dh1 in one launch; on the tcgen05 path it also writes the tf32 hi/lo pair noisy1_dgrad reads
    FinishNT jobs[2];
    for (int s = 0; s < 2; ++s)
      jobs[s] = make_finish_nt(&gb.p[s], 1, l->h1[0][s], l->dh1[s], true, l->um ? um_dh1_hi(l->um, s) : nullptr,
                               l->um ? um_dh1_lo(l->um, s) : nullptr);
    DZ_TRY(finish_nt_batch(jobs, 2, stream));
  }
  for (int s = 0; s < 2; ++s) {  // first noisy layer weight grads
    std::string pre = std::string(st[s]) + "1/";
    GemmProblem p = zero_problem();
    p.a_mode = A_PLAIN; p.A = l->act3[0]; p.lda = d.feat; p.M = B; p.K = d.feat;
    p.B = l->dh1[s]; p.N = 512; p.ldb = 512; p.ldc = 512;
    p.C = G + L.off(pre + "mu/w"); p.C2 = G + L.off(pre + "sigma/w"); p.Cb = G + L.off(pre + "mu/b"); p.Cb2 = G + L.off(pre + "sigma/b");
    p.a_scale = s == 0 ? nz.a1i : nz.v1i; p.c_scale = s == 0 ? nz.a1o : nz.v1o;
    gb.p[s] = p;
  }
  DZ_TRY(run_tn("noisy1_wgrad", gb, fork_side(l, stream)));
  if (l->um) {
    DZ_TRY(um_backward_fc(l->um, noise, stream));   // dh1 hi/lo came from the finish kernel above
    return DZ_OK;
  }
  for (int s = 0; s < 2; ++s) {  // dact3 contributions
    std::string pre = std::string(st[s]) + "1/";
    GemmProblem p = zero_problem();
    p.A = l->dh1[s]; p.lda = 512; p.M = B; p.N = 512; p.K = d.feat;
    p.B = P + L.off(pre + "mu/w"); p.B2 = P + L.off(pre + "sigma/w"); p.ldb = 512;
    p.a_scale = s == 0 ? nz.a1i : nz.v1i; p.c_scale = s == 0 ? nz.a1o : nz.v1o;
    p.ldc = d.feat;
    p.splits = l->nt_splits; p.split_stride = (long long)2 * B * d.feat;
    p.C = l->nt_partial + (long long)s * l->nt_splits * p.split_stride;
    gb.p[s] = p;
  }
  DZ_TRY(run_nt("noisy1_dgrad", gb, true, stream));
  // dact3 = (adv-stream + val-stream contributions) * [act3 > 0], summed from the split partials
  DZ_TRY(finish_nt(gb.p, 2, l->act3[0], l->dact3, true, stream));
  return DZ_OK;
}

int backward_iqn(dz_learner* l, void* stream) {
  const Dims& d = l->d;
  const Layout& L = l->lay;
  const dz_learner_config& c = l->cfg;
  const int B = l->B, N = l->n_head[0], M = B * N;
  float* G = l->buf.d_grads;
  const float* P = l->buf.d_online;
  GemmBatch gb;
  gb.n = 1;
  FinishTNBatch fb;
  fb.n = 0;
  float* part_head = l->tn_partial[3];
  float* part_embed = l->tn_partial[3] + (long long)16 * 513 * 64;
  {  // head wgrad: reduction over M rows
    GemmProblem p = zero_problem();
    p.a_mode = A_PLAIN; p.A = l->h1[0][0]; p.lda = 512; p.M = M; p.K = 512;
    p.B = l->dout; p.N = d.out; p.ldb = d.out; p.ldc = d.out;
    p.Cb = G + L.off("head/b");
    int splits = (int)std::min<int64_t>(16, ceil_div(M, 64));
    p.splits = splits; p.split_stride = (long long)513 * d.out; p.C = part_head;
    gb.p[0] = p;
    DZ_TRY(run_tn("iqn_head_wgrad", gb, fork_side(l, stream)));
    fb.f[fb.n++] = FinishTN{p.C, splits, p.split_stride, 512, d.out, G + L.off("head/w"), nullptr, p.Cb, nullptr, nullptr, nullptr};
  }
  {  // dh1
    GemmProblem p = zero_problem();
    p.A = l->dout; p.lda = d.out; p.M = M; p.N = d.out; p.K = 512;
    p.B = P + L.off("head/w"); p.ldb = d.out; p.C = l->dh1[0]; p.ldc = 512; p.mask = l->h1[0][0];
    gb.p[0] = p;
    if (M >= 512 && d.out <= kSkinnyMaxN) {
      DZ_LAUNCH_NAMED("iqn_head_dgrad", iqn_head_dgrad_kernel, (unsigned)std::min<int64_t>(ceil_div((long long)M * 128, 256), 148 * 8),
                      256, 0, stream, l->dout, P + L.off("head/w"), l->h1[0][0], l->dh1[0], M, d.out);
    } else {
      DZ_TRY(run_nt("iqn_head_dgrad", gb, false, stream));
    }
  }
  if (l->pk_on) {
    // dh1 in both operand orientations, then the two big contractions on the tcgen05 kernel
    PackBatch pb;
    memset(&pb, 0, sizeof(pb));
    DZ_TRY(pk_add_job(pb, l->dh1[0], 512, 0, 512, M, l->pk_dh1T.rows_pad, l->pk_dh1T.red_pad, -1, l->pk_dh1T.hi, l->pk_dh1T.lo));
    DZ_TRY(pk_add_job(pb, l->dh1[0], 512, 1, M, 512, l->pk_dh1.rows_pad, l->pk_dh1.red_pad, -1, l->pk_dh1.hi, l->pk_dh1.lo));
    if (l->pk_embed_bwd)   // cos^T plus a row of ones (bias gradient) for the embedding weight gradient
      DZ_TRY(pk_add_job(pb, l->cosf[0], c.latent_dim, 0, c.latent_dim, M, l->pk_cosT.rows_pad, l->pk_cosT.red_pad, c.latent_dim,
                        l->pk_cosT.hi, l->pk_cosT.lo));
    DZ_TRY(launch_pack("iqn_fc1_pack_bwd", pb, stream));
    PkBatch kb;
    memset(&kb, 0, sizeof(kb));
    kb.n = 1;
    kb.run_kb = 4;
    {  // fc1 wgrad: [feat + 1 (bias row), 512] = hi0^T(+ones) * dh1, reduction over the M rows, split partials
      PkProblem& p = kb.p[0];
      p.A = PkOperand{l->pk_actT.hi, l->pk_actT.lo, l->pk_actT.rows_pad / 8};
      p.B = PkOperand{l->pk_dh1T.hi, l->pk_dh1T.lo, l->pk_dh1T.rows_pad / 8};
      p.MI = d.feat + 1; p.NJ = 512; p.nkb = l->pk_actT.red_pad / kPkKB;
      p.sc_i = 512; p.sc_j = 1; p.splits = l->pk_wgrad_splits; p.split_stride = (long long)(d.feat + 1) * 512;
      p.C = l->pk_wgrad_partial;
      DZ_TRY(launch_pgemm("iqn_fc1_wgrad", kb, fork_side(l, stream)));
      fb.f[fb.n++] = FinishTN{p.C, p.splits, p.split_stride, d.feat, 512, G + L.off("fc1/w"), nullptr, G + L.off("fc1/b"), nullptr, nullptr, nullptr};
    }
    {  // dHI[m,k] = sum_n dh1[m,n] W[k,n]
      PkProblem& p = kb.p[0];
      memset(&p, 0, sizeof(p));   // (run_kb stays 4)
      p.A = PkOperand{l->pk_dh1.hi, l->pk_dh1.lo, l->pk_dh1.rows_pad / 8};
      p.B = PkOperand{l->pk_w.hi, l->pk_w.lo, l->pk_w.rows_pad / 8};
      p.MI = M; p.NJ = d.feat; p.nkb = l->pk_dh1.red_pad / kPkKB;
      p.sc_i = d.feat; p.sc_j = 1; p.splits = 1; p.split_stride = 0; p.C = l->dhi;
      DZ_TRY(launch_pgemm("iqn_fc1_dgrad", kb, stream));
    }
  } else {
  {  // fc1 wgrad (reduction over M rows, no split: 400 tiles already)
    GemmProblem p = zero_problem();
    p.a_mode = A_PLAIN; p.A = l->hi[0]; p.lda = d.feat; p.M = M; p.K = d.feat;
    p.B = l->dh1[0]; p.N = 512; p.ldb = 512; p.ldc = 512;
    p.C = G + L.off("fc1/w"); p.Cb = G + L.off("fc1/b");
    gb.p[0] = p;
    DZ_TRY(run_tn("iqn_fc1_wgrad", gb, fork_side(l, stream)));
  }
  {  // dHI = dh1 * Wf^T
    GemmProblem p = zero_problem();
    p.A = l->dh1[0]; p.lda = 512; p.M = M; p.N = 512; p.K = d.feat;
    p.B = P + L.off("fc1/w"); p.ldb = 512; p.C = l->dhi; p.ldc = d.feat;
    gb.p[0] = p;
    DZ_TRY(run_nt("iqn_fc1_dgrad", gb, false, stream));
  }
  }
  if (l->pk_embed_bwd) {
    dim3 hgrid((unsigned)(d.feat / 64), (unsigned)B);
    DZ_LAUNCH(iqn_hadamard_bwd_packed_kernel, hgrid, 256, 0, stream, l->dhi, l->E0, l->act3[0], l->dact3, l->pk_dET.hi,
              l->pk_dET.lo, l->pk_dET.rows_pad / 8, d.feat);
    // embed wgrad: [feat, latent + 1 (bias column)] = dE^T * [cos | 1], stored transposed into the [latent + 1, feat] partials
    PkBatch kb;
    memset(&kb, 0, sizeof(kb));
    kb.n = 1;
    kb.run_kb = 4;
    PkProblem& p = kb.p[0];
    p.A = PkOperand{l->pk_dET.hi, l->pk_dET.lo, l->pk_dET.rows_pad / 8};
    p.B = PkOperand{l->pk_cosT.hi, l->pk_cosT.lo, l->pk_cosT.rows_pad / 8};
    p.MI = d.feat; p.NJ = c.latent_dim + 1; p.nkb = l->pk_dET.red_pad / kPkKB;
    p.sc_i = 1; p.sc_j = d.feat; p.splits = l->pk_embed_wgrad_splits; p.split_stride = (long long)(c.latent_dim + 1) * d.feat;
    p.C = part_embed;
    DZ_TRY(launch_pgemm("iqn_embed_wgrad", kb, fork_side(l, stream)));
    fb.f[fb.n++] = FinishTN{p.C, p.splits, p.split_stride, c.latent_dim, d.feat, G + L.off("embed/w"), nullptr, G + L.off("embed/b"), nullptr, nullptr, nullptr};
  } else {
  DZ_LAUNCH(iqn_hadamard_bwd_kernel, (unsigned)ceil_div((long long)B * d.feat, 256), 256, 0, stream, l->dhi, l->E0, l->act3[0],
              l->dact3, B, N, d.feat);
    {  // embed wgrad: [latent, feat] = cos^T * dE
      GemmProblem p = zero_problem();
      p.a_mode = A_PLAIN; p.A = l->cosf[0]; p.lda = c.latent_dim; p.M = M; p.K = c.latent_dim;
      p.B = l->dhi; p.N = d.feat; p.ldb = d.feat; p.ldc = d.feat;
      p.Cb = G + L.off("embed/b");
      int splits = (int)std::min<int64_t>(16, ceil_div(M, 64));
      p.splits = splits; p.split_stride = (long long)(c.latent_dim + 1) * d.feat; p.C = part_embed;
      gb.p[0] = p;
      DZ_TRY(run_tn("iqn_embed_wgrad", gb, fork_side(l, stream)));
      fb.f[fb.n++] = FinishTN{p.C, splits, p.split_stride, c.latent_dim, d.feat, G + L.off("embed/w"), nullptr, p.Cb, nullptr, nullptr, nullptr};
    }
  }
  long long mx = 0;
  for (int q = 0; q < fb.n; ++q) mx = std::max<long long>(mx, (long long)(fb.f[q].K + 1) * fb.f[q].N);
  dim3 grid((unsigned)std::min<long long>(ceil_div(mx, 256), 148 * 8), fb.n);
  DZ_LAUNCH(finish_tn_kernel, grid, 256, 0, (l->side && l->side_dirty ? (void*)l->side : stream), fb);
  return DZ_OK;
}

// Split global norm (tcgen05 path, every agent but IQN): the sum of squares of everything behind the conv tensors is taken
// on the second side stream as soon as the last FC / head weight gradient is written (norm_fc_range), the conv tensors'
// partials come from the per-layer weight-gradient finish kernels, and the optimizer (or norm_finalize_kernel) combines them.
bool split_norm_active(const dz_learner* l) { return l->um != nullptr && l->cfg.kind != DZ_IQN && l->side2 != nullptr; }

int norm_fc_range(dz_learner* l, bool apply, void* stream) {
  const long long begin = l->lay.off(l->cfg.kind == DZ_RAINBOW ? "adv1/mu/w" : "fc1/w");
  const long long n = l->lay.total - begin;
  DZ_LAUNCH(grad_norm_kernel, kNormBlocks, 256, 0, stream, l->buf.d_grads + begin, n, l->scalars + 8, l->ticket, l->scalars + 1,
            apply ? l->buf.d_counters : l->buf.d_counters + 3, (float*)nullptr, 1);
  return DZ_OK;
}

int run_optimizer(dz_learner* l, float* user_norm, bool apply, void* stream) {
  const dz_learner_config& c = l->cfg;
  long long n = l->lay.total;
  float* norm = l->scalars;
  const bool split = split_norm_active(l);
  const float* parts = split ? l->norm_parts : nullptr;
  const int nparts = split ? um_norm_slots(l->um) : 0;
  if (!split) {
    DZ_LAUNCH(grad_norm_kernel, kNormBlocks, 256, 0, stream, l->buf.d_grads, n, l->scalars + 8, l->ticket, norm,
              apply ? l->buf.d_counters : l->buf.d_counters + 3, user_norm, 0);
  } else if (!apply) {
    DZ_LAUNCH(norm_finalize_kernel, 1, 256, 0, stream, parts, nparts, l->scalars + 1, norm, user_norm);
  }
  if (!apply) return DZ_OK;
  OptArgs o{c.optimizer, c.learning_rate, c.opt_eps, c.rms_decay, c.adam_b1, c.adam_b2, c.max_global_grad_norm,
            l->buf.d_online, l->buf.d_grads, l->buf.d_opt_state, l->buf.d_opt_state + n, n, norm, l->buf.d_counters,
            parts, nparts, l->scalars + 1, norm, user_norm};
  static const int per_sm = getenv("DZ_OPT_BLOCKS") ? atoi(getenv("DZ_OPT_BLOCKS")) : 8;
  // DZ_OPT_BULK=0: the register-staged kernel (A/B measurements)
  static const bool bulk = !(getenv("DZ_OPT_BULK") && getenv("DZ_OPT_BULK")[0] == '0');
  if (bulk) {
    static const int bulk_per_sm = getenv("DZ_OPT_BLOCKS") ? atoi(getenv("DZ_OPT_BLOCKS")) : 4;
    static const int stages = std::min(kOptStagesMax, std::max(2, getenv("DZ_OPT_STAGES") ? atoi(getenv("DZ_OPT_STAGES")) : 3));
    const int kOptSmem = stages * kOptStageBytes + 64;
    o.stages = stages;
    static const int vec = (getenv("DZ_OPT_VEC") && atoi(getenv("DZ_OPT_VEC")) == 4) ? 4 : 2;
    static bool attr_done = false;
    if (!attr_done) {
      DZ_CUDA_OK(cudaFuncSetAttribute(optimizer_bulk_kernel<DZ_ADAM, 4>, cudaFuncAttributeMaxDynamicSharedMemorySize, kOptSmem));
      DZ_CUDA_OK(cudaFuncSetAttribute(optimizer_bulk_kernel<DZ_RMSPROP_CENTERED, 4>, cudaFuncAttributeMaxDynamicSharedMemorySize, kOptSmem));
      DZ_CUDA_OK(cudaFuncSetAttribute(optimizer_bulk_kernel<DZ_ADAM, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, kOptSmem));
      DZ_CUDA_OK(cudaFuncSetAttribute(optimizer_bulk_kernel<DZ_RMSPROP_CENTERED, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, kOptSmem));
      attr_done = true;
    }
    const long long nchunks = ((o.n >> 2) + kOptChunk - 1) / kOptChunk;
    const unsigned grid = (unsigned)std::max<long long>(1, std::min<long long>(148LL * bulk_per_sm, nchunks));
    const unsigned threads = kOptChunk * 4 / vec;
    if (c.optimizer == DZ_ADAM) {
      if (vec == 4) DZ_LAUNCH_NAMED("optimizer_kernel", (optimizer_bulk_kernel<DZ_ADAM, 4>), grid, threads, kOptSmem, stream, o);
      else DZ_LAUNCH_NAMED("optimizer_kernel", (optimizer_bulk_kernel<DZ_ADAM, 2>), grid, threads, kOptSmem, stream, o);
    } else {
      if (vec == 4) DZ_LAUNCH_NAMED("optimizer_kernel", (optimizer_bulk_kernel<DZ_RMSPROP_CENTERED, 4>), grid, threads, kOptSmem, stream, o);
      else DZ_LAUNCH_NAMED("optimizer_kernel", (optimizer_bulk_kernel<DZ_RMSPROP_CENTERED, 2>), grid, threads, kOptSmem, stream, o);
    }
    return DZ_OK;
  }
  if (c.optimizer == DZ_ADAM) DZ_LAUNCH_NAMED("optimizer_kernel", optimizer_kernel<DZ_ADAM>, 148 * per_sm, 256, 0, stream, o);
  else DZ_LAUNCH_NAMED("optimizer_kernel", optimizer_kernel<DZ_RMSPROP_CENTERED>, 148 * per_sm, 256, 0, stream, o);
  return DZ_OK;
}

struct WriteBack { const dz_replay_view* view; const int64_t* indices; const float* priorities; double alpha; };

int update_impl(dz_learner* l, const dz_batch* batch, const dz_update_outputs* out, int apply_update, float* max_seen,
                const WriteBack* wb, void* stream, bool weights_packed = false) {
  const dz_learner_config& c = l->cfg;
  const Dims& d = l->d;
  const int B = l->B;
  const float* on = l->buf.d_online;
  const float* tg = l->buf.d_target;
  const bool needs_online_st = c.kind == DZ_DOUBLE_Q || c.kind == DZ_PRIORITIZED || c.kind == DZ_RAINBOW;
  if (c.kind == DZ_RAINBOW && !batch->d_noise) return fail(DZ_EINVAL, "rainbow update needs d_noise");
  if (c.kind == DZ_IQN && !batch->d_taus) return fail(DZ_EINVAL, "iqn update needs d_taus");
  if (!out || !out->d_loss || !out->d_per_example) return fail(DZ_EINVAL, "update outputs d_loss and d_per_example are required");
  if (!(weights_packed && l->um != nullptr)) DZ_TRY(join_side(l, stream));   // pending side-stream work (asynchronous randomness)

  // ---- forward: every network.apply of loss_fn in grouped launches
  TorsoJob jobs[3];
  int nj = 0;
  jobs[nj++] = TorsoJob{on, batch->d_s_tm1_rows, 0};
  if (needs_online_st) jobs[nj++] = TorsoJob{on, batch->d_s_t_rows, 1};
  jobs[nj++] = TorsoJob{tg, batch->d_s_t_rows, 2};
  const bool um = l->um != nullptr;
  if (um) {
    if (nj != l->um_npass) return fail(DZ_EINVAL, "tcgen05 path: pass count mismatch");
    const uint8_t* const* rows[3] = {nullptr, nullptr, nullptr};
    for (int i = 0; i < nj; ++i) rows[i] = jobs[i].rows;
    if (weights_packed) DZ_TRY(join_side(l, stream));   // packed on the side stream, concurrently with the sampler
    else DZ_TRY(um_pack_weights(l->um, stream));
    // Optional (DZ_PREFETCH=1): pull the 3136 -> 512 weight matrices into L2 beside the conv stack.  Measured on the
    // rainbow step: no gain (noisy1_fwd 23.0 vs 22.2 us, step 253 vs 244 us) — the layer is bound by its per-CTA pipeline,
    // not by DRAM — so it is off by default.
    static const bool prefetch = getenv("DZ_PREFETCH") != nullptr && getenv("DZ_PREFETCH")[0] == '1';
    if (prefetch && c.kind != DZ_IQN && l->side) DZ_TRY(um_prefetch_fc(l->um, fork_side(l, stream)));
    DZ_TRY(um_forward_torso(l->um, rows, stream));
    DZ_TRY(join_side(l, stream));
    if (c.kind != DZ_IQN) DZ_TRY(um_forward_fc(l->um, batch->d_noise, stream));
  } else {
    DZ_TRY(forward_torso(l, jobs, nj, B, stream));
  }

  if (c.kind == DZ_IQN) {
    // online(s_tm1, tau_tm1) | target(s_t, tau_selector) | target(s_t, tau_t)   (iqn/agent.py:192-203)
    Pass passes[3] = {{on, nullptr, 0, 0, 0}, {tg, nullptr, 2, 1, 0}, {tg, nullptr, 2, 2, 0}};
    const float* t0 = batch->d_taus;
    const float* t1 = t0 + (long long)B * c.tau_samples_s_tm1;
    const float* t2 = t1 + (long long)B * c.tau_samples_policy;
    const float* taus[3] = {t0, t1, t2};
    DZ_TRY(forward_heads_iqn(l, passes, 3, B, taus, true, stream));
  } else if (c.kind == DZ_RAINBOW) {
    Pass passes[3] = {{on, nullptr, 0, 0, 0}, {on, nullptr, 1, 1, 1}, {tg, nullptr, 2, 2, 2}};
    DZ_TRY(forward_heads_rainbow(l, passes, 3, B, batch->d_noise, stream, um));
  } else {
    Pass passes[3];
    int np = 0;
    passes[np++] = Pass{on, nullptr, 0, 0, 0};
    if (needs_online_st) passes[np++] = Pass{on, nullptr, 1, 1, 0};
    passes[np++] = Pass{tg, nullptr, 2, 2, 0};
    DZ_TRY(forward_heads_plain(l, passes, np, B, stream, um));
  }

  // ---- loss + gradient wrt the pass-0 head outputs
  LossArgs L;
  memset(&L, 0, sizeof(L));
  L.kind = c.kind; L.B = B; L.A = c.num_actions; L.atoms = c.num_atoms;
  L.out0 = l->out[0]; L.out1 = l->out[1]; L.out2 = l->out[2];
  L.adv0 = l->out[0]; L.val0 = l->outv[0]; L.adv1 = l->out[1]; L.val1 = l->outv[1]; L.adv2 = l->out[2]; L.val2 = l->outv[2];
  L.a = batch->d_a_tm1; L.r = batch->d_r_t; L.disc = batch->d_discount_t; L.w = batch->d_weights; L.taus0 = batch->d_taus;
  L.vmax = c.vmax; L.bound = c.grad_error_bound; L.kappa = c.huber_param;
  L.dout = l->dout; L.dadv = l->dout; L.dval = l->doutv;
  L.per_example = out->d_per_example; L.loss_terms = l->loss_terms;
  L.priorities = (c.kind == DZ_RAINBOW || c.kind == DZ_PRIORITIZED) ? out->d_priorities : nullptr;
  if (c.kind == DZ_DQN || c.kind == DZ_DOUBLE_Q || c.kind == DZ_PRIORITIZED) {
    DZ_LAUNCH(loss_q_kernel, B, 64, 0, stream, L);
  } else if (c.kind == DZ_C51 || c.kind == DZ_RAINBOW) {
    size_t smem = (6 * c.num_atoms + c.num_actions + 4) * sizeof(float);
    const size_t staged = (size_t)(c.num_atoms + 3 * c.num_actions * c.num_atoms + 3 * c.num_atoms) * sizeof(float);
    if (smem + staged <= 40 * 1024) DZ_LAUNCH_NAMED("loss_categorical_kernel", loss_categorical_staged_kernel, B, 128, smem + staged, stream, L);
    else DZ_LAUNCH(loss_categorical_kernel, B, 128, smem, stream, L);
  } else {
    if (c.kind == DZ_QRDQN) { L.N = c.num_quantiles; L.Ksel = c.num_quantiles; L.Nt = c.num_quantiles; }
    else { L.N = c.tau_samples_s_tm1; L.Ksel = c.tau_samples_policy; L.Nt = c.tau_samples_s_t; }
    size_t smem = (32 + c.num_actions + L.Nt + 2 * L.N) * sizeof(float);
    DZ_LAUNCH(loss_quantile_kernel, B, 256, smem, stream, L);
  }
  {   // the scalar loss / running max priority and replay.update_priorities(ids, priorities) (rainbow/agent.py:198) are
      // independent of the backward pass: both leave the critical path for the side stream
    void* ls = fork_side(l, stream);
    DZ_LAUNCH(loss_mean_kernel, 1, 32, 0, ls, l->loss_terms, B, out->d_loss, max_seen, L.priorities);
    if (wb) DZ_TRY(launch_update_priorities(wb->view, wb->indices, wb->priorities, B, wb->alpha, wb->view->capacity, ls));
  }

  // ---- backward through online(s_tm1)
  if (c.kind == DZ_RAINBOW) DZ_TRY(backward_rainbow(l, batch->d_noise, stream));
  else if (c.kind == DZ_IQN) DZ_TRY(backward_iqn(l, stream));
  else DZ_TRY(backward_plain(l, stream));
  if (split_norm_active(l)) {   // every gradient behind the conv tensors is final once the side stream's FC / head wgrads are done
    void* from = l->side_dirty ? (void*)l->side : stream;
    DZ_TRY(norm_fc_range(l, apply_update != 0, fork_side2(l, from, stream)));
  }
  DZ_TRY(backward_torso(l, batch->d_s_tm1_rows, stream));

  // ---- clip_by_global_norm + adam / rmsprop + apply_updates
  DZ_TRY(join_side2(l, stream));
  DZ_TRY(join_side(l, stream));
  DZ_TRY(run_optimizer(l, out->d_grad_norm, apply_update != 0, stream));
  return DZ_OK;
}

}  // namespace

// ------------------------------------------------------------------------------------------------
// C ABI
// ------------------------------------------------------------------------------------------------

extern "C" {

int dz_learner_plan_query(const dz_learner_config* cfg, dz_learner_plan* out) {
  DZ_TRY(validate(*cfg));
  dz_learner tmp;
  tmp.um = nullptr;
  memset(&tmp.buf, 0, sizeof(tmp.buf));
  tmp.cfg = *cfg;
  tmp.lay = make_layout(*cfg);
  tmp.d = make_dims(*cfg);
  tmp.B = cfg->batch;
  out->param_count = tmp.lay.total;
  out->num_tensors = (int32_t)tmp.lay.t.size();
  out->opt_state_floats = 2 * tmp.lay.total;
  read_env();
  out->workspace_bytes = carve(&tmp, nullptr);
  out->noise_floats = cfg->kind == DZ_RAINBOW ? 3 * noise_stride(*cfg, tmp.d) : 0;
  out->tau_floats = cfg->kind == DZ_IQN
                        ? (int64_t)cfg->batch * (cfg->tau_samples_s_tm1 + cfg->tau_samples_policy + cfg->tau_samples_s_t)
                        : 0;
  return DZ_OK;
}

int dz_learner_tensor_info(const dz_learner_config* cfg, int32_t i, char* name64, int64_t* shape4, int32_t* ndim, int64_t* offset) {
  DZ_TRY(validate(*cfg));
  Layout L = make_layout(*cfg);
  if (i < 0 || i >= (int)L.t.size()) return fail(DZ_ERANGE, "tensor index out of range");
  const TensorInfo& t = L.t[i];
  snprintf(name64, 64, "%s", t.name.c_str());
  for (int k = 0; k < 4; ++k) shape4[k] = t.shape[k];
  *ndim = t.ndim;
  *offset = t.offset;
  return DZ_OK;
}

int dz_learner_create(const dz_learner_config* cfg, const dz_learner_buffers* buf, dz_learner** out) {
  DZ_TRY(validate(*cfg));
  if (!buf->d_online || !buf->d_target || !buf->d_grads || !buf->d_opt_state || !buf->d_workspace || !buf->d_counters)
    return fail(DZ_EINVAL, "all learner buffers are required");
  read_env();
  dz_learner* l = new dz_learner();
  l->cfg = *cfg;
  l->buf = *buf;
  l->lay = make_layout(*cfg);
  l->d = make_dims(*cfg);
  l->B = cfg->batch;
  l->um = nullptr;
  carve(l, static_cast<char*>(buf->d_workspace));
  if (l->um_ws) {
    UmNetDesc ud = make_um_desc(l);
    int rc = um_net_create(ud, l->um_ws, &l->um);
    if (rc != DZ_OK) { delete l; return rc; }
    const bool three = ud.npass == 3;
    l->um_npass = ud.npass;
    l->um_set[0] = 0; l->um_set[1] = three ? 1 : 2; l->um_set[2] = 2;
    for (int i = 0; i < ud.npass; ++i) {   // the fp32 views the remaining FMA kernels, the losses and the tests read
      const int set = l->um_set[i];
      l->act1[set] = um_act_f32(l->um, 1, i); l->act2[set] = um_act_f32(l->um, 2, i); l->act3[set] = um_act_f32(l->um, 3, i);
      if (ud.use_fc)
        for (int s = 0; s < ud.nstream; ++s) l->h1[set][s] = um_h1_f32(l->um, i, s);
    }
    if (ud.use_fc)
      for (int s = 0; s < ud.nstream; ++s) l->dh1[s] = um_dh1_f32(l->um, s);
    l->dact3 = um_dact_f32(l->um, 3); l->dact2 = um_dact_f32(l->um, 2); l->dact1 = um_dact_f32(l->um, 1);
  }
  l->side = nullptr; l->ev_fork = nullptr; l->ev_join = nullptr; l->side_dirty = false;
  l->side2 = nullptr; l->ev_fork2 = nullptr; l->ev_join2 = nullptr; l->side2_dirty = false;
  if (getenv("DZ_NO_SIDE_STREAM") == nullptr) {
    if (cudaStreamCreateWithFlags(&l->side, cudaStreamNonBlocking) != cudaSuccess ||
        cudaEventCreateWithFlags(&l->ev_fork, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&l->ev_join, cudaEventDisableTiming) != cudaSuccess) {
      l->side = nullptr;
      cudaGetLastError();
    }
    if (l->side && (cudaStreamCreateWithFlags(&l->side2, cudaStreamNonBlocking) != cudaSuccess ||
                    cudaEventCreateWithFlags(&l->ev_fork2, cudaEventDisableTiming) != cudaSuccess ||
                    cudaEventCreateWithFlags(&l->ev_join2, cudaEventDisableTiming) != cudaSuccess)) {
      l->side2 = nullptr;
      cudaGetLastError();
    }
  }
  if (l->pk_on) {
    // fused epilogues only write the valid region of these images: zero the padding once, and set the constant
    // row of ones (bias-gradient row) of the transposed activation image
    for (int p = 0; p < 3; ++p) {
      cudaMemset(l->pk_act[p].hi, 0, pk_image_floats(l->pk_act[p].rows_pad, l->pk_act[p].red_pad) * sizeof(float));
      cudaMemset(l->pk_act[p].lo, 0, pk_image_floats(l->pk_act[p].rows_pad, l->pk_act[p].red_pad) * sizeof(float));
    }
    cudaMemset(l->pk_actT.hi, 0, pk_image_floats(l->pk_actT.rows_pad, l->pk_actT.red_pad) * sizeof(float));
    cudaMemset(l->pk_actT.lo, 0, pk_image_floats(l->pk_actT.rows_pad, l->pk_actT.red_pad) * sizeof(float));
    if (l->pk_embed_bwd) {
      cudaMemset(l->pk_dET.hi, 0, pk_image_floats(l->pk_dET.rows_pad, l->pk_dET.red_pad) * sizeof(float));
      cudaMemset(l->pk_dET.lo, 0, pk_image_floats(l->pk_dET.rows_pad, l->pk_dET.red_pad) * sizeof(float));
    }
    int rc = pk_set_ones_row(l->pk_actT.hi, l->pk_actT.rows_pad, l->d.feat, l->B * l->n_head[0], nullptr);
    if (rc != DZ_OK || cudaDeviceSynchronize() != cudaSuccess) { delete l; return rc != DZ_OK ? rc : fail(DZ_ECUDA, "packed image init"); }
  }
  cudaError_t e = cudaMemset(l->ticket, 0, 16);
  if (e != cudaSuccess) { delete l; return fail(DZ_ECUDA, "cudaMemset: %s", cudaGetErrorString(e)); }
  *out = l;
  return DZ_OK;
}

void dz_learner_destroy(dz_learner* l) {
  if (!l) return;
  um_net_destroy(l->um);
  if (l->side) { cudaStreamSynchronize(l->side); cudaStreamDestroy(l->side); }
  if (l->side2) { cudaStreamSynchronize(l->side2); cudaStreamDestroy(l->side2); }
  if (l->ev_fork) cudaEventDestroy(l->ev_fork);
  if (l->ev_join) cudaEventDestroy(l->ev_join);
  delete l;
}

int dz_learner_update(dz_learner* l, const dz_batch* batch, const dz_update_outputs* out, int32_t apply_update, void* stream) {
  return update_impl(l, batch, out, apply_update, nullptr, nullptr, stream);
}

int dz_learner_learn(dz_learner* l, const dz_replay_view* replay, int32_t prioritized, const dz_learn_io* io, void* stream) {
  const int B = l->B;
  BatchExtras ex{l->rows_sample[0], l->rows_sample[1], l->s_a, l->s_r, l->s_d, prioritized ? l->s_w : nullptr, 1};
  if (replay->obs_bytes != (int64_t)l->d.H * l->d.W * l->d.C) return fail(DZ_EINVAL, "replay observation size does not match the network");
  const bool frames = frame_store_on(replay);
  if (frames && (B > replay->frames.batch_capacity || !replay->frames.d_batch_stage))
    return fail(DZ_EINVAL, "batch exceeds the frame store's reserved batch staging");
  // conv weight images do not depend on the sampled batch: pack them on the side stream while the sampler runs
  const bool pack_aside = l->um != nullptr && l->side != nullptr;
  if (pack_aside) {
    void* ws = fork_side(l, stream);
    DZ_TRY(um_pack_weights(l->um, ws));
  }
  DZ_TRY(launch_sample(replay, prioritized, &io->sample_in, &io->sample_out, B, ex, stream));
  if (frames) {   // the row tables point at the staging rows; fill them from the sampled rows' frame slots
    uint8_t* stage = replay->frames.d_batch_stage;
    DZ_TRY(launch_frame_assemble(replay, io->sample_out.d_slots, B, stage,
                                 stage + (int64_t)replay->frames.batch_capacity * replay->obs_stride, replay->obs_stride, stream));
  }
  dz_batch batch;
  batch.d_s_tm1_rows = l->rows_sample[0];
  batch.d_s_t_rows = l->rows_sample[1];
  batch.d_a_tm1 = l->s_a; batch.d_r_t = l->s_r; batch.d_discount_t = l->s_d;
  batch.d_weights = prioritized ? l->s_w : nullptr;
  batch.d_taus = io->d_taus; batch.d_noise = io->d_noise;
  WriteBack wb{replay, io->sample_out.d_indices, io->update_out.d_priorities, io->priority_exponent};
  if (prioritized && !io->update_out.d_priorities) return fail(DZ_EINVAL, "prioritized learn needs update_out.d_priorities");
  DZ_TRY(update_impl(l, &batch, &io->update_out, 1, io->d_max_seen_priority, prioritized ? &wb : nullptr, stream, pack_aside));
  return DZ_OK;
}

// Same as dz_learner_generate_randomness, but enqueued on the learner's side stream (when it has one): the draws do not
// depend on the sampled batch, so they run beside the sampler instead of in front of it.  Ordered after everything already
// enqueued on `stream` and before the next dz_learner_learn / dz_learner_update / dz_learner_q_values on `stream`; any
// other consumer of the buffers must synchronise the device first.
int dz_learner_generate_randomness_async(dz_learner* l, uint64_t seed, float* d_taus, float* d_noise, void* stream) {
  return dz_learner_generate_randomness(l, seed, d_taus, d_noise, fork_side(l, stream));
}

int dz_learner_generate_randomness(dz_learner* l, uint64_t seed, float* d_taus, float* d_noise, void* stream) {
  const dz_learner_config& c = l->cfg;
  if (c.kind == DZ_IQN && d_taus) {
    long long n = (long long)c.batch * (c.tau_samples_s_tm1 + c.tau_samples_policy + c.tau_samples_s_t);
    DZ_LAUNCH(randomness_kernel, (unsigned)ceil_div(ceil_div(n, 4), 256), 256, 0, stream, d_taus, n, seed, l->buf.d_counters, 0, 1u);
  }
  if (c.kind == DZ_RAINBOW && d_noise) {
    long long n = 3 * noise_stride(c, l->d);
    DZ_LAUNCH(randomness_kernel, (unsigned)ceil_div(ceil_div(n, 4), 256), 256, 0, stream, d_noise, n, seed, l->buf.d_counters, 1, 2u);
  }
  DZ_LAUNCH(bump_counter_kernel, 1, 1, 0, stream, l->buf.d_counters, 1);
  return DZ_OK;
}

int dz_learner_q_values(dz_learner* l, const uint8_t* d_obs, const float* d_taus, const float* d_noise, float* d_q_out, void* stream) {
  const dz_learner_config& c = l->cfg;
  const float* on = l->buf.d_online;
  DZ_TRY(join_side(l, stream));   // pending side-stream work (asynchronous randomness)
  DZ_LAUNCH(make_row_table_kernel, 1, 32, 0, stream, d_obs, (long long)0, 1, l->rows_act);
  TorsoJob job{on, l->rows_act, 1};   // use activation set 1 so a pending backward's set-0 buffers stay intact
  DZ_TRY(forward_torso(l, &job, 1, 1, stream));
  Pass pass{on, nullptr, 1, 1, 0};
  int nq = 1;
  if (c.kind == DZ_IQN) {
    if (!d_taus) return fail(DZ_EINVAL, "iqn q_values needs taus[tau_samples_policy]");
    const float* taus[1] = {d_taus};
    DZ_TRY(forward_heads_iqn(l, &pass, 1, 1, taus, false, stream));
    nq = c.tau_samples_policy;
  } else if (c.kind == DZ_RAINBOW) {
    if (!d_noise) return fail(DZ_EINVAL, "rainbow q_values needs one apply of noise");
    DZ_TRY(forward_heads_rainbow(l, &pass, 1, 1, d_noise, stream));
  } else {
    DZ_TRY(forward_heads_plain(l, &pass, 1, 1, stream));
    nq = c.num_quantiles;
  }
  size_t smem = (32 + c.num_atoms + 8) * sizeof(float);
  DZ_LAUNCH(q_values_kernel, 1, 128, smem, stream, c.kind, c.num_actions, c.num_atoms, nq, c.vmax, l->out[1], l->out[1], l->outv[1], d_q_out);
  return DZ_OK;
}

// Batched acting (parts.py:342-411 with many actors; dqn/agent.py:121-131,169-177): online forward on E <= batch observations
// in one enqueue, q-values [E][A], and the epsilon-greedy choice on the device — one D2H of E actions per tick instead of a
// D2H sync per decision.  d_obs: E contiguous observations (H*W*C bytes each).  d_explore: [2][E] uniforms in [0,1) or
// NULL (greedy): action = u0 < epsilon ? floor(u1 * A) : argmax (first maximum, as np.argmax).  IQN: d_taus is
// [E][tau_samples_policy]; rainbow: ONE noise apply shared by the E streams of the tick (the reference's actors each draw
// their own: statistically the same exploration, not the same sample path).
int dz_learner_act_batch(dz_learner* l, const uint8_t* d_obs, int32_t E, const float* d_taus, const float* d_noise,
                         const float* d_explore, float epsilon, float* d_q_out, int32_t* d_actions, void* stream) {
  const dz_learner_config& c = l->cfg;
  const float* on = l->buf.d_online;
  if (E < 1 || E > l->B) return fail(DZ_EINVAL, "act_batch: 1 <= E <= learner batch");
  if (!d_obs || !d_q_out || !d_actions) return fail(DZ_EINVAL, "act_batch: null buffer");
  DZ_TRY(join_side(l, stream));
  const long long obs_bytes = (long long)l->d.H * l->d.W * l->d.C;
  DZ_LAUNCH(make_row_table_kernel, (unsigned)ceil_div(E, 64), 64, 0, stream, d_obs, obs_bytes, (int)E, l->rows_act);
  TorsoJob job{on, l->rows_act, 1};
  DZ_TRY(forward_torso(l, &job, 1, E, stream));
  Pass pass{on, nullptr, 1, 1, 0};
  int nq = 1;
  if (c.kind == DZ_IQN) {
    if (!d_taus) return fail(DZ_EINVAL, "iqn act_batch needs taus[E][tau_samples_policy]");
    const float* taus[1] = {d_taus};
    DZ_TRY(forward_heads_iqn(l, &pass, 1, E, taus, false, stream));
    nq = c.tau_samples_policy;
  } else if (c.kind == DZ_RAINBOW) {
    if (!d_noise) return fail(DZ_EINVAL, "rainbow act_batch needs one apply of noise");
    DZ_TRY(forward_heads_rainbow(l, &pass, 1, E, d_noise, stream));
  } else {
    DZ_TRY(forward_heads_plain(l, &pass, 1, E, stream));
    nq = c.num_quantiles;
  }
  size_t smem = (32 + c.num_atoms + 8) * sizeof(float);
  DZ_LAUNCH(q_values_kernel, (unsigned)E, 128, smem, stream, c.kind, c.num_actions, c.num_atoms, nq, c.vmax, l->out[1], l->out[1], l->outv[1], d_q_out);
  DZ_LAUNCH(act_select_kernel, (unsigned)ceil_div(E, 128), 128, 0, stream, (const float*)d_q_out, c.num_actions, (int)E, d_explore, epsilon, d_actions);
  return DZ_OK;
}

namespace {
__global__ void u8_to_unit_table_kernel(float* out) {
  dz::pdl_enter();
  out[threadIdx.x] = u8_to_unit(threadIdx.x);
}
}  // namespace

// Test hook: the device's uint8 -> float32/255 conversion of 0..255 (the conv1 operand load of the fp32-FMA kernels).
int dz_test_u8_to_unit(float* d_out256, void* stream) {
  DZ_LAUNCH(u8_to_unit_table_kernel, 1, 256, 0, stream, d_out256);
  return DZ_OK;
}

int dz_learner_sync_target(dz_learner* l, void* stream) {
  DZ_CUDA_OK(cudaMemcpyAsync(l->buf.d_target, l->buf.d_online, l->lay.total * sizeof(float), cudaMemcpyDeviceToDevice,
                             (cudaStream_t)stream));
  return DZ_OK;
}

// Debug hook: the tcgen05 launch named `tag` ("conv2_fwd", "conv3_fwd", "fc1_fwd", "fc1_dgrad", "conv3_dgrad", "conv2_dgrad",
// "conv3_wgrad", "conv2_wgrad") writes the clock stamps of its CTA 0 into d_trace (512 int64); nullptr switches it off.
int dz_test_learner_trace(dz_learner* l, const char* tag, long long* d_trace) {
  if (!l->um) return fail(DZ_EINVAL, "the tcgen05 path is not active for this learner");
  um_net_trace(l->um, tag, d_trace);
  return DZ_OK;
}

// Test hook: device-to-device copy out of an internal buffer (tests hold only the raw pointer).
int dz_test_copy(void* d_dst, const void* d_src, int64_t bytes, void* stream) {
  DZ_CUDA_OK(cudaMemcpyAsync(d_dst, d_src, (size_t)bytes, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  return DZ_OK;
}

// Test hook: device pointer + element count of an internal activation / gradient buffer (tests and tools only).
int dz_test_learner_buffer(dz_learner* l, const char* name, float** d_ptr, int64_t* count) {
  const std::string n = name;
  const int64_t rows0 = (int64_t)l->B * l->n_head[0];
  if (n == "act3") { *d_ptr = l->act3[0]; *count = (int64_t)l->B * l->d.feat; }
  else if (n == "act1") { *d_ptr = l->act1[0]; *count = (int64_t)l->B * l->d.h1 * l->d.w1 * 32; }
  else if (n == "act2") { *d_ptr = l->act2[0]; *count = (int64_t)l->B * l->d.h2 * l->d.w2 * 64; }
  else if (n == "h1_val") { *d_ptr = l->h1[0][1]; *count = l->h1[0][1] ? rows0 * 512 : 0; }
  else if (n == "iqn_e0") { *d_ptr = l->E0; *count = l->E0 ? rows0 * l->d.feat : 0; }
  else if (n == "h1") { *d_ptr = l->h1[0][0]; *count = rows0 * 512; }
  else if (n == "dh1") { *d_ptr = l->dh1[0]; *count = rows0 * 512; }
  else if (n == "iqn_hi") {
    if (l->pk_on) return fail(DZ_EINVAL, "iqn_hi is not materialised on the packed tcgen05 path (DZ_PK_IQN=0 keeps it)");
    *d_ptr = l->hi[0]; *count = l->hi[0] ? rows0 * l->d.feat : 0;
  }
  else if (n == "iqn_dhi") { *d_ptr = l->dhi; *count = l->dhi ? rows0 * l->d.feat : 0; }
  else return fail(DZ_EINVAL, "unknown buffer '%s'", name);
  if (!*d_ptr) return fail(DZ_EINVAL, "buffer '%s' is not used by this agent kind", name);
  return DZ_OK;
}

}  // extern "C"
