// Internal (non-ABI) interfaces between affinity.cu (exact scan, orchestration) and affinity_f16.cu
// (FP16 candidate filter over the key image, threshold select, exact re-rank).
#pragma once
#include "common.cuh"

namespace cutie {

struct RerankParams {
  KeySegments segs;
  const float* qk;
  const float* qe;
  long long Q, n_total;
  const int* cand_idx;
  const int* count;
  int cap, top_k, kpad;
  int* out_idx;
  float* out_w;
  float* out_sim;
  unsigned long long* usage_acc;
};

// FP16 filter over the key operand image (affinity_f16.cu): threshold sampling pass + candidate filter pass.
constexpr int F16_RESERVE = 16;            // candidate slots reserved per global atomic (per thread)
constexpr int F16_SLOTS = 8;               // running minima per sampling thread (threshold slots = splits x 2 x F16_SLOTS)
struct F16FilterParams {
  KeySegments segs;
  const float* qk;
  const float* qe;
  const float* key_mu;             // [B][64] centre the image was built with (null = 0): the operand uses qk - mu
  long long Q;
  // sample pass: tiles g = tile_phase + j * tile_stride of the image; output group_min [B][Q][groups_per_query]
  int tile_stride, tile_phase;
  float* group_min;
  int groups_per_query;
  // filter pass: thresholds in, per-query candidate lists out
  const float* emax_in;
  int* cand_idx;
  int* count;
  int cap;
  // CTA schedule (f16_schedule)
  int full_groups, splits_full, splits_half;
  // per segment: the FP16 operand image of the arena it lives in (cutie_bank_key_image), by physical 128-token tile
  const unsigned char* img[kMaxSeg];
  long long img_bs[kMaxSeg];       // batch stride (bytes)
  long long img_tile0[kMaxSeg];    // first physical tile of the segment
  int img_lo0[kMaxSeg];            // row of the segment's first token inside that tile
  long long img_tcum[kMaxSeg + 1]; // prefix sums of the segments' tile counts
};
size_t f16_filter_smem_bytes();
int f16_schedule(F16FilterParams& p, long long B);
int launch_f16_filter(const F16FilterParams& p, long long B, int grid_x, bool sample, cudaStream_t st);
struct F16ThresholdParams {
  const float* group_min;      // [B][Q][groups] slot minima of the sample pass
  int groups, top_k, kpad;
  long long Q, n_total;
  float* emax_out;             // [B][Q]
  // optional seeds: [B][Q][kpad] token indices (first top_k entries; -1 = none), evaluated exactly against this query
  const int* seed_idx;
  KeySegments segs;
  const float* qk;
  const float* qe;
};
int launch_f16_threshold(const F16ThresholdParams& p, long long B, cudaStream_t st);

int launch_rerank(const RerankParams& p, long long B, cudaStream_t st);

}  // namespace cutie
