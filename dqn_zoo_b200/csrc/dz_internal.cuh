// Internal (non-ABI) declarations shared between the replay and learner translation units.
#pragma once
#include "dz_common.cuh"

namespace dz {

// Optional per-batch outputs the fused learner path wants straight from the sampler:
// row pointers into the replay store (the gather is fused into the conv1 operand load) and the
// float32/int32 scalars exactly as they enter jit(update).
struct BatchExtras {
  const uint8_t** d_s_tm1_rows;
  const uint8_t** d_s_t_rows;
  int32_t* d_a;
  float* d_r;
  float* d_disc;
  float* d_w;
  int fused;
};

int launch_sample(const dz_replay_view* view, int prioritized, const dz_sample_inputs* in, const dz_sample_outputs* out,
                  int batch, const BatchExtras& ex, void* stream);
int launch_update_priorities(const dz_replay_view* view, const int64_t* d_indices, const float* d_priorities, int n,
                             double alpha, int64_t size, void* stream);
int launch_fill_scalars(const dz_replay_view* view, int64_t row0, int64_t n, uint64_t seed, int num_actions,
                        double discount, void* stream);

// ---- frame-deduplicated storage (dz_frames.cu) ------------------------------------------------------------------
bool frame_store_on(const dz_replay_view* v);
// Every argument check of frames_insert; dz_replay_add runs it before it enqueues anything for the add.
int frames_check_add(const dz_replay_view* v, const dz_add_record* rec);
// The insert of one add whose two stacks are already in v->frames.d_add_stage.
int frames_insert(const dz_replay_view* v, const dz_add_record* rec, void* stream);
// HWC stacks of rows d_slots[0..batch): s_tm1 of row b at dst0 + b * pitch, s_t at dst1 + b * pitch.
int launch_frame_assemble(const dz_replay_view* v, const int64_t* d_slots, int batch, uint8_t* dst0, uint8_t* dst1,
                          int64_t pitch, void* stream);


// ---- packed-operand tcgen05 GEMM (dz_tcp.cuh / dz_tcp.cu) ------------------------------------------------------
constexpr int kPkKB = 16;         // reduction elements per k-block / pipeline stage
constexpr int kPkMaxJobs = 8;
constexpr int kPkMaxProblems = 4;

struct PackJob {
  const float* src;
  int ld;
  int red_contig;          // 1: element (row, r) at src[row * ld + r];  0: at src[r * ld + row]
  int rows, red;           // valid extents (everything outside reads as zero)
  int rows_pad, red_pad;   // image extents
  int ones_row;            // row index that reads as 1.0 for every valid r (bias-gradient row), or -1
  float* hi;
  float* lo;
  int tiles_r;             // 64-row tiles per 64-deep slab
  int block0;              // first block of this job in the flattened grid
};
struct PackBatch { PackJob job[kPkMaxJobs]; int n; int blocks; };

struct PkOperand { const float* hi; const float* lo; int rg_total; };   // rg_total = rows_pad / 8
struct PkProblem {
  PkOperand A, B;          // A: 128-row tiles (rows i), B: BNJ-row tiles (rows j)
  int MI, NJ, nkb;         // nkb = red_pad / 16
  float* C;                // partial s at C + s * split_stride; element (i,j) at i * sc_i + j * sc_j
  long long sc_i, sc_j, split_stride;
  int splits;
  const float* bias_j;     // splits == 1 only: + bias_j[j], then optional ReLU
  int relu;
  // EPI 1 (IQN embedding epilogue; dz_tcp.cuh): v = relu(acc + bias_j[j]) -> e0[i * e0_ld + j] (optional);
  // h = v * mul[(i / mul_div) * mul_ld + j] -> hi/lo images with rows i (img_*) and optionally rows j (imgT_*)
  float* e0; int e0_ld;
  const float* mul; int mul_div, mul_ld;
  float *img_hi, *img_lo; int img_rg;
  float *imgT_hi, *imgT_lo; int imgT_rg;
};
struct PkBatch { PkProblem p[kPkMaxProblems]; int n; int run_kb; };   // run_kb: k-blocks per accumulation run (0: default 4)


inline int64_t pk_image_floats(int rows_pad, int red_pad) { return (int64_t)rows_pad * red_pad; }
int pk_add_job(PackBatch& pb, const float* src, int ld, int red_contig, int rows, int red, int rows_pad, int red_pad,
               int ones_row, float* hi, float* lo);
int launch_pack(const char* tag, const PackBatch& pb, void* stream);
int pk_set_ones_row(float* hi, int rows_pad, int row, int red, void* stream);   // image element (row, r < red) = 1
int launch_pgemm(const char* tag, const PkBatch& kb, void* stream, int epi = 0);

}  // namespace dz
