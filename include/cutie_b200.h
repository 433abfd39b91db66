/*
 * cutie_b200.h -- C-ABI of libcutie_b200.so: hand-written sm_100a kernels for the Cutie per-frame
 * hot path (pixel-memory readout + object-transformer attention).
 *
 * The reference (hkchengrex/Cutie) has no FFI layer: its "operator interface" for this path is a set
 * of Python functions/methods that call PyTorch library kernels.  Each entry point below names the
 * reference call site(s) it replaces (paths relative to the reference root).  A replacement
 * implementation must export exactly these symbols; cutie_b200/kernels.py binds them with ctypes and
 * INTEGRATION.md shows the reference-side binding a maintainer would add.
 *
 * Conventions
 *   - plain pointers + int64 sizes/strides (strides in ELEMENTS); no torch types cross this boundary;
 *   - every buffer (inputs, outputs, workspaces) is allocated and owned by the caller; kernels borrow
 *     pointers for the duration of the enqueued work and never allocate;
 *   - all work is enqueued on `stream` (a cudaStream_t passed as void*); nothing synchronises;
 *   - return 0 on success, <0 on invalid argument (-1) or launch failure (-2); never throws;
 *     cutie_b200_last_error() returns a thread-local message for the last failure;
 *   - all floating point is fp32 (the reference runs this path with amp=False, eval_config.yaml:13);
 *   - "token-major" = [B, n, C] with the channel axis contiguous (one memory token per row);
 *     "channel-major" = [B, C, n] as PyTorch convolutions emit feature maps.
 */
#ifndef CUTIE_B200_H_
#define CUTIE_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CUTIE_B200_ABI_VERSION 2
#define CUTIE_B200_MAX_SEGMENTS 4       /* long | permanent | ring piece a | ring piece b */
#define CUTIE_B200_USAGE_FRAC_BITS 40   /* usage accumulators: uint64 fixed point, 2^-40 */

int cutie_b200_abi_version(void);
const char* cutie_b200_last_error(void);

/* ---- pixel-memory readout ------------------------------------------------------------------------ */

/* Fused similarity -> exact top-k -> softmax over the winners.
 * Replaces get_similarity (cutie/model/utils/memory_utils.py:7-46) + do_softmax(top_k=..., return_usage)
 * (memory_utils.py:49-77) as called from MemoryManager.read (cutie/inference/memory_manager.py:144-172),
 * including the torch.cat of long-term and working keys (:137-143): the bank is passed as up to 4
 * token-major segments, indices count tokens across segments in order.
 *   S[n,q] = -shrinkage[n]/sqrt(CK) * sum_c qe[c,q] * (key[n,c] - qk[c,q])^2      (== memory_utils.py:28-42)
 *   out_idx/out_w [B,Q,kpad]: the top_k tokens per query by (S desc, index asc) and exp(S)/sum exp(S) over
 *   them; slots >= top_k hold (-1, 0).  out_sim (optional) the winners' S.  usage_acc (optional, uint64
 *   [B, n_total], zeroed by the caller) += w * 2^40 per winner (deterministic integer accumulation of
 *   memory_utils.py:74-75).
 * CK must be 64; top_k <= kpad, kpad in {32, 64}. */
size_t cutie_affinity_workspace_bytes(int64_t B, int64_t Q, int64_t n_total, int top_k);
int cutie_affinity_topk(int num_segments, const void* const* seg_key, const void* const* seg_shrinkage,
                        const int64_t* seg_len, const int64_t* seg_key_bstride, const int64_t* seg_shr_bstride,
                        const float* qk, const float* qe, int64_t B, int64_t CK, int64_t Q, int top_k, int kpad,
                        int32_t* out_idx, float* out_w, float* out_sim, unsigned long long* usage_acc,
                        int64_t n_total, void* workspace, size_t workspace_bytes, void* stream);
/* Same call with the bank's precomputed FP16 tcgen05 operand image (cutie_bank_key_image): seg_key_image[s] is the
 * image of the ARENA segment s lives in ([B, tiles, 9216] floats = 36864 bytes of f16 operands per 128-token tile,
 * batch stride seg_image_bstride[s]), seg_phys_begin[s] the segment's first token's index inside that arena, key_mu
 * ([B, 64] or NULL) the key centre every one of those images was built with.  With images the call runs the FP16 plan
 * (csrc/affinity_f16.cu): tile-sampled threshold pass, threshold select, candidate filter over the whole image (one
 * 36 KB cp.async.bulk per tile), exact fp32 re-rank; the outputs are bit-identical to cutie_affinity_topk.
 * seed_idx ([B, Q, kpad] or NULL): per query top_k DISTINCT token indices (e.g. the previous frame's winners) whose
 * exact energies tighten the filter threshold; they never change the result, only how many candidates are re-ranked.
 * seg_key_image == NULL (or a NULL entry for a non-empty segment) = no images: the exact fp32 scan, at every bank size. */
int cutie_affinity_topk_img(int num_segments, const void* const* seg_key, const void* const* seg_shrinkage,
                            const int64_t* seg_len, const int64_t* seg_key_bstride, const int64_t* seg_shr_bstride,
                            const void* const* seg_key_image, const int64_t* seg_image_bstride,
                            const int64_t* seg_phys_begin, const float* key_mu, const int32_t* seed_idx, const float* qk,
                            const float* qe, int64_t B, int64_t CK,
                            int64_t Q, int top_k, int kpad, int32_t* out_idx, float* out_w, float* out_sim,
                            unsigned long long* usage_acc, int64_t n_total, void* workspace,
                            size_t workspace_bytes, void* stream);

/* Execution plan of cutie_affinity_topk_img for a bank of n_total tokens when every segment carries a key image:
 * 0 = exact fp32 scan; 1 = the FP16 filter plan (csrc/affinity_f16.cu) followed by an exact fp32 re-rank of the
 * survivors.  A call without images always runs plan 0.  Both plans return the same selection and weights (the
 * filter only discards tokens that provably cannot be in the top-k).
 * cutie_set_tc_min_tokens: banks smaller than n use plan 0 (default 6144; negative restores the default). */
int cutie_affinity_plan(int64_t n_total, int top_k);
/* Diagnostics: byte offset of the per-query candidate counters inside the workspace of a filtered call (-1: exact scan). */
int64_t cutie_debug_ws_count_offset(int64_t B, int64_t Q, int64_t n_total, int top_k);
void cutie_set_tc_min_tokens(int64_t n);
/* Diagnostics: per-phase device times (ms) of the filtered plan's launches (sample pass, threshold select, filter
 * pass, exact re-rank) for one of the last 64 calls, measured in situ with events on the caller's stream. */
void cutie_debug_phase_timing(int enable);
int cutie_debug_phase_times(int64_t calls_ago, float* out_ms, int max_phases);
/* Number of filter passes served from a key image so far in this process (diagnostics / tests). */
int64_t cutie_debug_image_level_launches(void);

/* Merge `nparts` sorted candidate lists per query (part_val/part_idx [B, nparts, Q, kpad], unused slots
 * idx = INT32_MAX or -1 with val = -inf) into the global top_k + softmax; same outputs as cutie_affinity_topk.
 * Used by the key-sharded multi-GPU read after the NCCL all-gather of per-shard candidates (SURVEY.md 8(e).2);
 * there is no reference counterpart (the reference is single-GPU). */
int cutie_topk_merge(const float* part_val, const int32_t* part_idx, int64_t B, int64_t nparts, int64_t Q,
                     int top_k, int kpad, int32_t* out_idx, float* out_w, float* out_sim,
                     unsigned long long* usage_acc, int64_t n_total, void* stream);

/* Sparse value readout out[b,k,c,q] = sum_j w[b,q,j] * V_k[idx[b,q,j], c].
 * Replaces MemoryManager._readout (memory_manager.py:77-88; dense [K*CV,N]x[N,Q] GEMM against a matrix
 * with top_k non-zeros per column) and _get_visual_values_by_ids (:101-110; torch.stack/cat of the whole
 * value bank every frame).  seg_val[s*K + k] -> token-major values of object k in segment s. */
int cutie_readout_gather(const int32_t* idx, const float* w, int64_t B, int64_t Q, int kpad, int num_segments,
                         const int64_t* seg_len, const void* const* seg_val, const int64_t* seg_val_bstride,
                         int64_t K, int64_t CV, float* out, void* stream);

/* use_cnt += usage_acc * 2^-40 ; life_cnt += 1  for n tokens.
 * Replaces KeyValueMemoryStore.update_bucket_usage (cutie/inference/kv_memory_store.py:151-162). */
int cutie_usage_commit(float* use_cnt, int64_t use_bstride, float* life_cnt, int64_t life_bstride,
                       const unsigned long long* usage_acc, int64_t acc_bstride, int64_t acc_offset, int64_t B,
                       int64_t n, void* stream);

/* ---- mask decoder glue ------------------------------------------------------------------------------- */

/* out[b,k,c] = bilinear_x2(g[b,k,c]) + skip[b,c]   (align_corners = False), g [B,K,C,h,w], skip [B,C,2h,2w],
 * out [B,K,C,2h,2w], all contiguous.  Replaces UpsampleBlock's F.interpolate + broadcast add
 * (cutie/model/modules.py:15-19, group_modules.py:11-24 upsample_groups) on the frame path. */
int cutie_upsample2x_add(const float* g, const float* skip, float* out, int64_t B, int64_t K, int64_t C, int64_t h,
                         int64_t w, void* stream);

/* y = act(y + bias[c] (+ z)) in place, act = ReLU if `relu` else identity: the epilogue of a convolution called
 * without its bias.  Replaces the broadcast bias add inside every `nn.Conv2d` call on the frame path plus the
 * `F.relu` / residual `+` that follow it in the reference's blocks (cutie/model/group_modules.py:46-64 GroupResBlock,
 * cutie/model/channel_attn.py:27-38 CAResBlock, cutie/model/utils/resnet.py:77-131 BasicBlock/Bottleneck,
 * cutie/model/big_modules.py:64-87 KeyProjection ...).  y (and z, if not null) dense fp32 [N,C,HW] when
 * channels_last == 0, [N,HW,C] when 1; bias [C].  Association as in ATen: (y + bias) + z, then the clamp. */
int cutie_bias_act(float* y, const float* bias, const float* z, int64_t N, int64_t C, int64_t HW, int channels_last,
                   int relu, void* stream);

/* out[p,Y,X] = mean of the f x f window of in[p]: F.interpolate(mode='area') / adaptive_avg_pool2d for sizes that
 * divide (H % f == 0, W % f == 0).  Replaces the 16x mask down-sampling of CUTIE.pixel_fusion (cutie/model/cutie.py:149),
 * the 2x / 4x feature down-sampling of SensoryUpdater (cutie/model/modules.py:58-60, group_modules.py:27-36
 * downsample_groups) and ObjectSummarizer's mask resize (object_summarizer.py:60).  in [planes,H,W], out
 * [planes,H/f,W/f], dense fp32; row-major fp32 accumulation, one division. */
int cutie_area_pool(const float* in, float* out, int64_t planes, int64_t H, int64_t W, int64_t f, void* stream);

/* CAResBlock tail (cutie/model/channel_attn.py:27-38): gate[n,c] = sigmoid(conv1d_k(mean[n,:])[c]) (zero padded, no
 * bias), then y = y * gate + x in place.  y, x dense fp32 [N,C,HW] (channels_last == 0) or [N,HW,C] (1); mean [N,C] =
 * spatial mean of y (caller supplied); w [k], k odd; gate [N,C] scratch. */
int cutie_eca_scale_add(float* y, const float* x, const float* mean, const float* w, float* gate, int64_t N, int64_t C,
                        int64_t HW, int64_t k, int channels_last, void* stream);

/* Sensory GRU update (cutie/model/modules.py:37-45 _recurrent_update): v [P,3d,HW] = [forget | update | candidate],
 * h [P,d,HW] -> out [P,d,HW] = sigmoid(vf) * h * (1 - sigmoid(vu)) + sigmoid(vu) * tanh(vn).  Dense fp32. */
int cutie_gated_update(const float* v, const float* h, float* out, int64_t P, int64_t d, int64_t HW, void* stream);

/* out = relu(maxpool3x3/stride2/pad1(y) + bias[c]) == maxpool(relu(y + bias)): the tail of both ResNet stems
 * (cutie/model/utils/resnet.py:139-142; cutie/model/big_modules.py:42-46, 150-154) applied to the BIAS-LESS
 * convolution output (BatchNorm folded).  y [N,C,H,W] dense fp32 (channels_last == 0) or [N,H,W,C] (1, needs
 * C % 4 == 0), out the same layout with Ho = (H-1)/2 + 1, Wo = (W-1)/2 + 1. */
int cutie_bias_relu_maxpool(const float* y, const float* bias, float* out, int64_t N, int64_t C, int64_t H, int64_t W,
                            int channels_last, void* stream);

/* CUTIE.segment tail (cutie/model/cutie.py:196-203; aggregate cutie/utils/tensor_utils.py:47-54): x [B,K,h,w] decoder
 * logits at stride 4 -> agg [B,1+K,h,w] = log-odds of clamp([prod(1-sigmoid x) | sigmoid x], 1e-7, 1-1e-7) (scratch /
 * by-product), logits [B,1+K,4h,4w] = bilinear x4 (align_corners = False) of agg, prob = softmax over the 1+K channels.
 * K <= 15; all dense fp32. */
int cutie_segment_tail(const float* x, float* agg, float* logits, float* prob, int64_t B, int64_t K, int64_t h, int64_t w,
                       void* stream);

/* 3x3 (zero-pad 1) and 1x1 convolutions, stride 1 or 2, as tcgen05 implicit GEMMs with 3xTF32 operand splitting
 * (fp32-class accuracy, measured 2-6x closer to float64 than cuDNN's fp32 result; csrc/conv_tc.cu):
 *     y = act(bias + conv(pre(x), W) [+ residual]),  pre = ReLU if relu_in, act = ReLU if relu_out.
 * x [NB, Cin, H_in, W_in], y / residual [NB, Cout, H_out, W_out] fp32, each addressed through three ELEMENT strides
 * {image, channel, pixel} (pixel = row * width + column): dense NCHW = {C*H*W, H*W, 1}, channels-last = {C*H*W, 1, C}.
 * Cin % 32 == 0; output channels are processed in tiles of 128 (a partial last tile costs a full one).
 * Replaces the F.conv2d calls of PixelFFN / CAResBlock (transformer_layers.py:121-136, channel_attn.py:7-39),
 * PixelFeatureFuser (big_modules.py:192-235), KeyProjection (big_modules.py:66-87), MaskDecoder / SensoryUpdater
 * (big_modules.py:238-306, modules.py:46-85) and the 3x3 and 1x1 convolutions of the ResNet trunks
 * (utils/resnet.py:77-131) -- SURVEY.md section 8(f).1-3.
 * `weight_image` is the layer's operand image: cutie_conv_weight_image(weight [Cout, Cin, k, k]) once per weight version,
 * cutie_conv_weight_image_bytes(Cout, Cin, k) bytes (tf32 hi | lo planes per (128-channel tile, 32-channel chunk, tap) in
 * K-major SWIZZLE_128B order: one 32 KB cp.async.bulk per MMA step). */
int64_t cutie_conv_weight_image_bytes(int64_t Cout, int64_t Cin, int ksize);
int cutie_conv_weight_image(const float* weight, int64_t Cout, int64_t Cin, int ksize, void* image, void* stream);
int cutie_conv_tc(const float* x, const int64_t* x_strides, const void* weight_image, const float* bias,
                  const float* residual, const int64_t* residual_strides, int64_t NB, int64_t Cin, int64_t Cout,
                  int64_t H_in, int64_t W_in, int ksize, int stride, int relu_in, int relu_out, float* y,
                  const int64_t* y_strides, int units_per_cta, float* workspace, int32_t* counters, void* stream);
/* Launch plan of cutie_conv_tc: out6 = {output tiles T (images x 128-channel tiles x spatial tiles), MMA N, input chunks C per
 * tile, (tile, chunk) units per CTA q, CTAs, workspace floats}.  CTA i owns units [i q, (i + 1) q) of the T x C space (any
 * q <= C is valid: a share spans at most two tiles): layers with at least as many tiles as SMs run one whole tile per CTA
 * (q = C, no workspace); smaller layers split every tile uniformly over input-channel ranges (q = C / s, the largest s <= 8
 * with CTAs <= SMs); the shares of a tile meet in `workspace` and the CTA that arrives last adds them in slot order
 * (deterministic) before the epilogue.  `counters` (T int32) must be zero on entry
 * and are zero again on exit.  units_per_cta = 0: the plan's choice (pass the same value to both calls). */
int cutie_conv_plan(int64_t NB, int64_t Cin, int64_t Cout, int64_t H_in, int64_t W_in, int ksize, int stride, int units_per_cta,
                    int64_t* out6);
/* test hook: the spatial tile the launcher picks (out3 = {rows, columns, MMA N}). */
int cutie_debug_conv_tile_shape(int64_t H, int64_t W, int* out3);

/* 3x3 convolution with a single output channel, optionally of the rectified input: the mask decoder's prediction head
 * `pred(F.relu(p4))` (cutie/model/big_modules.py:264,300; Conv2d(C, 1, 3, padding=1)).  x [planes,C,H,W] dense fp32
 * (planes = B*K objects), w [C,3,3] (= weight[0]), bias [1], out [planes,H,W]; zero padding of the (rectified) input. */
int cutie_conv3x3_c1(const float* x, const float* w, const float* bias, float* out, int64_t planes, int64_t C, int64_t H,
                     int64_t W, int relu_input, void* stream);

/* out[y,x] = lut[argmax_c prob[c,y,x]]: InferenceCore.output_prob_to_mask (inference_core.py:377-385: argmax over
 * the 1+K channels, then ObjectManager.tmp_to_obj_cls object_manager.py:99-104) in one pass.  prob may be a strided
 * view (plane_stride / row_stride in elements, unit pixel stride); lut int64 [C]; out int64 [H,W] contiguous.
 * Ties: the first maximum wins (torch.argmax); NaN is not treated specially. */
int cutie_prob_to_mask(const float* prob, int64_t plane_stride, int64_t row_stride, int64_t C, int64_t H, int64_t W,
                       const int64_t* lut, int64_t* out, void* stream);

/* ---- memory bank maintenance ------------------------------------------------------------------------ */

/* dst[b,i,c] = src[b,c,i]  (channel-major feature map -> token-major arena rows).
 * Replaces the flatten + torch.cat growth of KeyValueMemoryStore.add (kv_memory_store.py:6-16,:136-149). */
int cutie_bank_append(const float* src, int64_t src_bstride, float* dst_rows, int64_t dst_bstride, int64_t B,
                      int64_t C, int64_t n, void* stream);
/* Build / refresh the FP16 tcgen05 operand image for tokens [phys_begin, phys_begin + n) of an arena (key_arena
 * [B, cap, 64], shr_arena [B, cap] token-major; image [B, image_tiles, 9216] floats, image_tiles*128 >= cap; key_mu [B, 64] or NULL: the image holds k - mu.
 * Tile t of the image holds tokens [128 t, 128 t + 128) as 36864 bytes of f16 operands [shr k^2 | shr k | error-bound
 * tail] in the filter's shared-memory layout (2 SWIZZLE_128B K-blocks + tail; csrc/tc_operand_f16.cuh).
 * Called once per memory frame for the appended tokens -- the per-token part of get_similarity
 * (memory_utils.py:28-36: mk^2, shrinkage scaling) hoisted out of the per-frame read; no reference counterpart. */
int cutie_bank_key_image(const float* key_arena, int64_t key_bstride, const float* shr_arena, int64_t shr_bstride,
                         int64_t B, int64_t phys_begin, int64_t n, float* image, int64_t image_bstride,
                         int64_t image_tiles, const float* key_mu, void* stream);
/* dst[b,c,i] = rows[b,i,c]  (token-major -> channel-major; reference-shaped views for inspection). */
int cutie_bank_export(const float* rows, int64_t rows_bstride, float* dst, int64_t dst_bstride, int64_t B,
                      int64_t C, int64_t n, void* stream);
/* dst_rows[b,j,:] = concat(segments)[b, index[b,j], :].  Replaces the advanced-index gathers of
 * remove_obsolete_features (kv_memory_store.py:226-242) and consolidation (memory_manager.py:340-344). */
int cutie_bank_gather(int num_segments, const void* const* seg_rows, const int64_t* seg_len,
                      const int64_t* seg_bstride, const int64_t* index, float* dst_rows, int64_t dst_bstride,
                      int64_t B, int64_t m, int64_t C, void* stream);
/* Long-term potentiation: for every prototype p, A[:,p] = softmax_n(S[n,p]) over ALL candidate tokens
 * (max-subtracted, memory_utils.py:68-71), out_val_k[b,p,:] = sum_n A[n,p] V_k[n,:], out_shr[b,p] = sum_n A[n,p] shr[n].
 * Replaces MemoryManager.consolidation (memory_manager.py:345-356).  workspace: B*P*n_total floats. */
int cutie_consolidate(int num_segments, const void* const* seg_key, const void* const* seg_shrinkage,
                      const int64_t* seg_len, const int64_t* seg_key_bstride, const int64_t* seg_shr_bstride,
                      const void* const* seg_val, const int64_t* seg_val_bstride, int64_t K,
                      const float* proto_key, int64_t pk_bstride, const float* proto_sel, int64_t ps_bstride,
                      int64_t B, int64_t P, int64_t CK, int64_t CV, void* const* out_val,
                      const int64_t* out_val_bstride, float* out_shr, int64_t out_shr_bstride, float* workspace,
                      int64_t n_total, void* stream);
/* The same potentiation over ONE SHARD of the candidates (key-sharded memory, cutie_b200/inference/sharded.py): results are
 * normalised by the shard's own statistics, which are also returned -- out_max[b,p] = max_n S[n,p] (the per-shard affinity
 * maximum BASELINE.json's north_star exchanges), out_sumexp[b,p] = sum_n exp(S[n,p] - out_max[b,p]) -- so that the shards'
 * results combine exactly like one softmax: weight_r = sumexp_r exp(max_r - M) / sum_r' (...), M = max_r max_r.
 * Both null: identical to cutie_consolidate.  (memory_manager.py:345-356, memory_utils.py:68-71.) */
int cutie_consolidate_partial(int num_segments, const void* const* seg_key, const void* const* seg_shrinkage,
                              const int64_t* seg_len, const int64_t* seg_key_bstride, const int64_t* seg_shr_bstride,
                              const void* const* seg_val, const int64_t* seg_val_bstride, int64_t K,
                              const float* proto_key, int64_t pk_bstride, const float* proto_sel, int64_t ps_bstride,
                              int64_t B, int64_t P, int64_t CK, int64_t CV, void* const* out_val,
                              const int64_t* out_val_bstride, float* out_shr, int64_t out_shr_bstride, float* out_max,
                              float* out_sumexp, float* workspace, int64_t n_total, void* stream);
/* acc[i] += add[i].  Replaces the streaming object-memory sum (memory_manager.py:252-271). */
int cutie_obj_summary_accumulate(float* acc, const float* add, int64_t n, void* stream);

/* ---- object transformer ----------------------------------------------------------------------------- */

/* Skinny fused linear on the [M = B*K*16, Kd] query tile:
 *   xin = x  (or x[:, :Kd] / (x[:, Kd] + 1e-4) when summary_norm: row stride Kd+1; object_transformer.py:126-132)
 *   xin = LayerNorm(xin) * ln_w + ln_b   (Kd == 256; xhat_out <- this)           transformer_layers.py:34,75,115
 *   xin += pe                                                                      transformer_layers.py:36,77
 *   y = xin . W^T + bias ; relu ; y += residual[(m % residual_mod) or m]           nn.Linear / in_proj / out_proj
 * Replaces the addmm/layer_norm/add/relu ATen launches of SelfAttention, CrossAttention, FFN
 * (transformer_layers.py:12-118) and the query initialisation (object_transformer.py:133-138). */
int cutie_qt_linear(const float* x, int64_t M, int64_t Kd, const float* W, int64_t ldw, int64_t N,
                    const float* bias, const float* ln_w, const float* ln_b, const float* pe, int summary_norm,
                    int relu, const float* residual, int64_t residual_mod, float* xhat_out, float* y, void* stream);
/* out[m,h,c] = scale * sum_d a[m, h*dh+d] * Wx[h*dh+d, c]  (Wx = W or W^T), dots[m,h] = scale * a_h . bias_h.
 * Folds one side's per-head projection into the other side's input space so the per-pixel K/V (or Q/out)
 * projections of nn.MultiheadAttention (transformer_layers.py:88-93) never run. */
int cutie_qt_head_fold(const float* a, int64_t M, int64_t E, int num_heads, const float* W, int64_t ldw,
                       int transpose_w, float scale, const float* bias_vec, float* out, float* dots, void* stream);
/* 16x16 self attention per (object, head): SelfAttention core (transformer_layers.py:40). */
int cutie_qt_self_attention(const float* qk, const float* v, int64_t M, int64_t E, int num_queries, int num_heads,
                            float* out, void* stream);
/* The query-side chain of the object transformer as ONE launch (csrc/qt.cu, qt_chain_kernel): an op list over the
 * [objects x 16, 256] query tile -- the same ops, with the same arguments, as cutie_qt_linear / cutie_qt_head_fold /
 * cutie_qt_self_attention and the merge step of cutie_qt_pixel_to_query -- executed by a persistent grid.  Ops that share a
 * `phase` are independent of each other; a grid barrier separates consecutive phases, so an op may read what ops of EARLIER
 * phases wrote.  Results are bit-identical to the separate launches.  Replaces the addmm / layer_norm / SDPA launches of
 * QueryTransformerBlock.forward between the two cross attentions (object_transformer.py:46-68, transformer_layers.py:12-118).
 *   LINEAR          in = {x, W, bias, ln_w, ln_b, pe, residual}  out = {y, xhat_out}
 *                   i = {M, Kd, ldw, N, flags (1 = summary_norm, 2 = relu), residual_mod}
 *   HEAD_FOLD       in = {a, W, bias_vec}  out = {out, dots}  i = {M, ldw, transpose_w}  f = scale
 *   SELF_ATTENTION  in = {qk, v}  out = {out}  i = {M}
 *   P2Q_COMBINE     in = {workspace of cutie_qt_pixel_to_query(attn_out = NULL), wv, bv}  out = {attn}  i = {tiles, ldwv, BK}
 * prefetch_ptr / prefetch_bytes: read-only ranges (weights) to pull into L2 at the start.  sync_ws: 4 uint32, zero before
 * the first launch and owned by ONE stream at a time (the kernel leaves them zero). */
enum { CUTIE_QT_OP_LINEAR = 0, CUTIE_QT_OP_HEAD_FOLD = 1, CUTIE_QT_OP_SELF_ATTENTION = 2, CUTIE_QT_OP_P2Q_COMBINE = 3 };
#define CUTIE_QT_CHAIN_MAX_OPS 16
#define CUTIE_QT_CHAIN_MAX_PREFETCH 16
typedef struct cutie_qt_op {
  int32_t kind, phase;
  const float* in[8];
  float* out[2];
  int64_t i[6];
  float f;
  int32_t reserved;
} cutie_qt_op;
int cutie_qt_chain(const cutie_qt_op* ops, int nops, const void* const* prefetch_ptr, const int64_t* prefetch_bytes,
                   int nprefetch, uint32_t* sync_ws, void* stream);
/* mask_pred 1x1 conv on relu(pixel) + sigmoid + aggregate + foreground test + per-object foreground count.
 * Replaces mask_pred[i] and QueryTransformer._get_aux_mask (object_transformer.py:153-155,165-167,179-205;
 * cutie/utils/tensor_utils.py:47-54).  The [(B*K*heads),Q,HW] bool mask is represented by fg + fg_count. */
int cutie_qt_aux_mask(const float* pixel, const float* w, const float* b, int64_t B, int64_t K, int64_t E,
                      int64_t HW, float* logits, uint8_t* fg, int32_t* fg_count, void* stream);
/* read_from_pixel attention core (masked, queries <- pixels) on tcgen05 tensor cores (3xTF32, fp32-class accuracy):
 * one CTA per 64-pixel tile and object computes S = Qfold.(pixel+pe), the masked tile-local softmax and Z = P.pixel^T
 * (csrc/qt_tc.cu); a combine kernel merges the tiles and applies the per-head value projection.  Replaces
 * CrossAttention.cross_attn for read_from_pixel (transformer_layers.py:88-93 via object_transformer.py:51-56).
 * `splits` must be cutie_qt_pixel_to_query_splits() = ceil(HW/64); workspace: cutie_qt_pixel_to_query_workspace_floats(). */
int cutie_qt_pixel_to_query_splits(int64_t BK, int64_t HW, int num_heads);
int64_t cutie_qt_pixel_to_query_workspace_floats(int64_t BK, int64_t HW);
int cutie_qt_pixel_to_query(const float* qfold, const float* pixel, const float* pixel_pe, const uint8_t* fg,
                            const int32_t* fg_count, const float* wv, int64_t ldwv, const float* bv, int64_t BK,
                            int64_t E, int64_t HW, int num_queries, int num_heads, int splits, float* workspace,
                            float* attn_out, void* stream);
/* read_from_query (pixels <- queries) on tcgen05 tensor cores (3xTF32): one CTA per 128-pixel tile and object, fused
 * through the per-head softmax over the 16 queries, value fold, output bias and residual, channel-major in/out.  Replaces CrossAttention for read_from_query (object_transformer.py:61-65) and the
 * NLC<->NCHW permutes around it (:50, transformer_layers.py:131-132). */
int cutie_qt_query_to_pixel(const float* kfold, const float* kdots, const float* vfold, const float* out_bias,
                            const float* pixel, const float* pixel_pe, int64_t BK, int64_t E, int64_t HW,
                            int num_queries, int num_heads, float* out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* CUTIE_B200_H_ */
