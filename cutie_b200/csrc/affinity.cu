// Pixel-memory readout for sm_100a: similarity scan + exact streaming top-k, split merge + softmax,
// sparse value gather.  See include/cutie_b200.h for the contract and DESIGN.md for the roofline.
//
// Kernel 1  affinity_scan_kernel   grid (query tiles of 64, key splits, B), 256 threads, ~204 KB smem
//   Streams its split of the memory bank through a 2-stage cp.async pipeline of 128-token tiles
//   (token-major rows, 256 B each, padded to 272 B in smem so LDS.128 is conflict free), evaluates
//   S[n,q] = -shr[n]/sqrt(CK) * sum_c (a[q,c]*k[n,c] - b[q,c])^2 with a = sqrt(qe), b = a*qk
//   (2 FFMA per channel; cancellation free, unlike the reference's 3-term expansion), filters against
//   the per-query running k-th best, and pushes survivors into a CTA queue that the warps drain into
//   per-query sorted lists.  The [N,HW] similarity matrix never exists.
// Kernel 2  topk_merge_kernel      one warp per query: merges the per-split sorted lists, softmax over
//   the winners, optional fixed-point usage accumulation (deterministic).
// Kernel 3  readout_gather_kernel  one warp per query x object: gathers the k winning 1 KB value rows,
//   accumulates in registers, transposes through smem to the channel-major [B,K,CV,Q] output.
#include "topk_common.cuh"
#include "affinity_internal.cuh"

namespace cutie {
thread_local char g_last_error[512] = "";

constexpr int TQ = 64;     // queries per CTA
constexpr int TK = 128;    // memory tokens per tile
constexpr int NT = 256;    // threads per CTA
constexpr int LDT = 68;    // padded smem row stride (floats)
constexpr int QCAP = TQ * TK;

struct ScanParams {
  KeySegments segs;
  const float* qk;
  const float* qe;
  long long Q;
  long long n_total;
  int top_k;
  int kpad;
  int tiles_per_split;
  int nsplit;
  float* part_val;  // [B][nsplit][Q][kpad]
  int* part_idx;
};

struct ScanSmem {
  float ks[2][TK][LDT];
  float as_[TQ][LDT];
  float bs_[TQ][LDT];
  unsigned long long queue[QCAP];
  float lval[TQ][KPAD_MAX];
  int lidx[TQ][KPAD_MAX];
  float sh[2][TK];
  float tau[TQ];
  int qcount[2];
};

__device__ __forceinline__ void load_key_tile(ScanSmem& sm, int stage, const ScanParams& p, int b, long long i0,
                                              long long i_end, int tid) {
  const int c4 = tid & 15;
#pragma unroll
  for (int it = 0; it < TK / 16; ++it) {
    int r = (tid >> 4) + 16 * it;
    long long i = i0 + r;
    float* dst = &sm.ks[stage][r][4 * c4];
    if (i < i_end) {
      int s = seg_of(p.segs.begin, p.segs.nseg, i);
      const float* src = p.segs.key[s] + (long long)b * p.segs.key_bs[s] + (i - p.segs.begin[s]) * CKD + 4 * c4;
      cp_async16(dst, src);
    } else {
      *reinterpret_cast<float4*>(dst) = make_float4(0.f, 0.f, 0.f, 0.f);
    }
  }
  if (tid < TK) {
    long long i = i0 + tid;
    if (i < i_end) {
      int s = seg_of(p.segs.begin, p.segs.nseg, i);
      cp_async4(&sm.sh[stage][tid], p.segs.shr[s] + (long long)b * p.segs.shr_bs[s] + (i - p.segs.begin[s]));
    } else {
      sm.sh[stage][tid] = 0.f;
    }
  }
}

template <int NS>
__global__ void __launch_bounds__(NT, 1) affinity_scan_kernel(const ScanParams p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  ScanSmem& sm = *reinterpret_cast<ScanSmem*>(smem_raw);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int b = blockIdx.z, split = blockIdx.y;
  const long long q0 = (long long)blockIdx.x * TQ;
  const long long split_begin = (long long)split * p.tiles_per_split * TK;
  long long split_end = split_begin + (long long)p.tiles_per_split * TK;
  if (split_end > p.n_total) split_end = p.n_total;
  const int ntiles = split_end > split_begin ? (int)((split_end - split_begin + TK - 1) / TK) : 0;
  const float scale = rsqrtf((float)CKD);

  // ---- prologue: query operands a = sqrt(qe), b = a*qk, transposed to [q][c]; empty lists ----
  for (int i = tid; i < CKD * TQ; i += NT) {
    int c = i / TQ, q = i % TQ;
    float e = 0.f, k = 0.f;
    if (q0 + q < p.Q) {
      long long off = ((long long)b * CKD + c) * p.Q + q0 + q;
      e = p.qe[off];
      k = p.qk[off];
    }
    float a = sqrtf(e);
    sm.as_[q][c] = a;
    sm.bs_[q][c] = a * k;
  }
  for (int i = tid; i < TQ * KPAD_MAX; i += NT) {
    (&sm.lval[0][0])[i] = -CUDART_INF_F;
    (&sm.lidx[0][0])[i] = INT_MAX;
  }
  if (tid < TQ) sm.tau[tid] = -CUDART_INF_F;
  if (tid < 2) sm.qcount[tid] = 0;
  if (ntiles > 0) load_key_tile(sm, 0, p, b, split_begin, split_end, tid);
  cp_async_commit();

  const int tn = tid & 15, tq = tid >> 4;
  for (int t = 0; t < ntiles; ++t) {
    const int st = t & 1;
    cp_async_wait<0>();
    __syncthreads();
    if (t + 1 < ntiles) load_key_tile(sm, st ^ 1, p, b, split_begin + (long long)(t + 1) * TK, split_end, tid);
    cp_async_commit();

    // ---- 8 tokens x 4 queries per thread ----
    float acc[8][4];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
#pragma unroll 4
    for (int c4 = 0; c4 < CKD / 4; ++c4) {
      float4 kf[8], af[4], bf[4];
#pragma unroll
      for (int i = 0; i < 8; ++i) kf[i] = *reinterpret_cast<const float4*>(&sm.ks[st][tn + 16 * i][4 * c4]);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        af[j] = *reinterpret_cast<const float4*>(&sm.as_[tq + 16 * j][4 * c4]);
        bf[j] = *reinterpret_cast<const float4*>(&sm.bs_[tq + 16 * j][4 * c4]);
      }
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          float d;
          d = fmaf(af[j].x, kf[i].x, -bf[j].x); acc[i][j] = fmaf(d, d, acc[i][j]);
          d = fmaf(af[j].y, kf[i].y, -bf[j].y); acc[i][j] = fmaf(d, d, acc[i][j]);
          d = fmaf(af[j].z, kf[i].z, -bf[j].z); acc[i][j] = fmaf(d, d, acc[i][j]);
          d = fmaf(af[j].w, kf[i].w, -bf[j].w); acc[i][j] = fmaf(d, d, acc[i][j]);
        }
    }
    // ---- threshold filter -> CTA queue ----
    float tauq[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) tauq[j] = sm.tau[tq + 16 * j];
    const long long tile_g0 = split_begin + (long long)t * TK;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int r = tn + 16 * i;
      const float sscale = -sm.sh[st][r] * scale;
      const bool valid = tile_g0 + r < split_end;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float s = acc[i][j] * sscale;
        const bool pass = valid && (q0 + tq + 16 * j < p.Q) && (s > tauq[j]);
        const unsigned m = __ballot_sync(0xffffffffu, pass);
        if (m) {
          int base = 0;
          if (lane == 0) base = atomicAdd(&sm.qcount[st], __popc(m));
          base = __shfl_sync(0xffffffffu, base, 0);
          if (pass) {
            const int slot = base + __popc(m & ((1u << lane) - 1u));
            const unsigned lo = ((unsigned)(tq + 16 * j) << 24) | (unsigned)(t * TK + r);
            sm.queue[slot] = ((unsigned long long)__float_as_uint(s) << 32) | lo;
          }
        }
      }
    }
    __syncthreads();
    // ---- drain: warp w owns queries q with q % 8 == w ----
    const int qn = sm.qcount[st];
    if (tid == 0) sm.qcount[st ^ 1] = 0;
    for (int base = 0; base < qn; base += 32) {
      const int e = base + lane;
      unsigned long long ent = 0ull;
      bool mine = false;
      if (e < qn) {
        ent = sm.queue[e];
        mine = (((unsigned)(ent >> 24) & 0xffu) & 7u) == (unsigned)warp;
      }
      unsigned bits = __ballot_sync(0xffffffffu, mine);
      while (bits) {
        const int src = __ffs(bits) - 1;
        bits &= bits - 1;
        const unsigned long long ce = __shfl_sync(0xffffffffu, ent, src);
        const float s = __uint_as_float((unsigned)(ce >> 32));
        const int ql = (int)((ce >> 24) & 0xffu);
        const int idx = (int)(split_begin + (long long)(ce & 0xffffffu));
        const float kth = sm.lval[ql][p.top_k - 1];
        if (s > kth || (s == kth && idx < sm.lidx[ql][p.top_k - 1])) {
          float tau = list_insert<NS>(&sm.lval[ql][0], &sm.lidx[ql][0], lane, p.top_k, s, idx);
          if (lane == 0) sm.tau[ql] = tau;
          __syncwarp();
        }
      }
    }
  }
  __syncthreads();
  // ---- write this split's sorted lists ----
  const int kp = p.kpad;
  for (int i = tid; i < TQ * kp; i += NT) {
    int q = i / kp, j = i % kp;
    if (q0 + q < p.Q) {
      long long o = (((long long)b * p.nsplit + split) * p.Q + q0 + q) * kp + j;
      p.part_val[o] = sm.lval[q][j];
      p.part_idx[o] = sm.lidx[q][j];
    }
  }
}

struct MergeParams {
  const float* part_val;
  const int* part_idx;
  long long Q;
  long long n_total;
  int nsplit, top_k, kpad;
  int* out_idx;
  float* out_w;
  float* out_sim;
  unsigned long long* usage_acc;
};

template <int NS>
__global__ void __launch_bounds__(256) topk_merge_kernel(const MergeParams p) {
  __shared__ float lv[8][KPAD_MAX];
  __shared__ int li[8][KPAD_MAX];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int b = blockIdx.y;
  const long long q = (long long)blockIdx.x * 8 + warp;
  if (q >= p.Q) return;
  const int kp = p.kpad;
  for (int u = 0; u < NS; ++u) { lv[warp][lane + 32 * u] = -CUDART_INF_F; li[warp][lane + 32 * u] = INT_MAX; }
  __syncwarp();
  // split 0 is already sorted: adopt it wholesale
  {
    const long long o = (((long long)b * p.nsplit) * p.Q + q) * kp;
    for (int u = 0; u < NS; ++u) {
      int slot = lane + 32 * u;
      if (slot < p.top_k) {
        const int ci = p.part_idx[o + slot];
        const bool dead = ci < 0 || ci == INT_MAX;          // -1 (public output format) or INT_MAX (scan lists)
        lv[warp][slot] = dead ? -CUDART_INF_F : p.part_val[o + slot];
        li[warp][slot] = dead ? INT_MAX : ci;
      }
    }
    __syncwarp();
  }
  for (int s = 1; s < p.nsplit; ++s) {
    const long long o = (((long long)b * p.nsplit + s) * p.Q + q) * kp;
    for (int j = 0; j < p.top_k; ++j) {
      const float cv = p.part_val[o + j];
      const int ci = p.part_idx[o + j];
      if (ci == INT_MAX || ci < 0) break;             // end of this split's list
      const float kth = lv[warp][p.top_k - 1];
      const int kthi = li[warp][p.top_k - 1];
      if (!(cv > kth || (cv == kth && ci < kthi))) break;   // sorted: the rest are worse too
      list_insert<NS>(&lv[warp][0], &li[warp][0], lane, p.top_k, cv, ci);
    }
  }
  const long long oo = ((long long)b * p.Q + q) * kp;
  finalize_topk<NS>(&lv[warp][0], &li[warp][0], lane, p.top_k, kp, p.out_idx + oo, p.out_w + oo,
                    p.out_sim ? p.out_sim + oo : nullptr,
                    p.usage_acc ? p.usage_acc + (long long)b * p.n_total : nullptr);
}

// ------------------------------------------------------------------------------------------------
struct GatherParams {
  const int* idx;
  const float* w;
  long long Q;
  int kpad;
  RowSegments segs;
  long long K, CV;
  float* out;
};

constexpr int GQ = 32;  // queries per CTA in the gather kernel

// CV == 256: each lane owns 8 channels (two float4) of the output row.
__global__ void __launch_bounds__(256) readout_gather_kernel(const GatherParams p) {
  __shared__ float tile[256][GQ + 1];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int k = blockIdx.y, b = blockIdx.z;
  const long long q0 = (long long)blockIdx.x * GQ;
  const int ns = p.kpad / 32;
  for (int qi = warp; qi < GQ; qi += 8) {
    const long long q = q0 + qi;
    float4 a0 = make_float4(0.f, 0.f, 0.f, 0.f), a1 = a0;
    if (q < p.Q) {
      const long long o = ((long long)b * p.Q + q) * p.kpad;
      for (int u = 0; u < ns; ++u) {
        const int myi = p.idx[o + lane + 32 * u];
        const float myw = p.w[o + lane + 32 * u];
        unsigned livem = __ballot_sync(0xffffffffu, myi >= 0);   // holes allowed (sharded banks own a subset)
        while (livem) {
          // up to 4 winners per trip so several 1 KB row reads are in flight
          int js[4];
          int cnt = 0;
#pragma unroll
          for (int t = 0; t < 4; ++t) {
            if (livem) { js[t] = __ffs(livem) - 1; livem &= livem - 1; ++cnt; } else { js[t] = -1; }
          }
          float4 v0[4], v1[4];
          float wj[4];
#pragma unroll
          for (int t = 0; t < 4; ++t) {
            if (t < cnt) {
              const int id = __shfl_sync(0xffffffffu, myi, js[t]);
              wj[t] = __shfl_sync(0xffffffffu, myw, js[t]);
              const int s = seg_of(p.segs.begin, p.segs.nseg, id);
              const float* row = p.segs.rows[s * p.segs.nobj + k] + (long long)b * p.segs.bs[s * p.segs.nobj + k] +
                                 ((long long)id - p.segs.begin[s]) * 256;
              v0[t] = __ldg(reinterpret_cast<const float4*>(row) + lane);
              v1[t] = __ldg(reinterpret_cast<const float4*>(row) + 32 + lane);
            }
          }
#pragma unroll
          for (int t = 0; t < 4; ++t) {
            if (t < cnt) {
              a0.x = fmaf(wj[t], v0[t].x, a0.x); a0.y = fmaf(wj[t], v0[t].y, a0.y);
              a0.z = fmaf(wj[t], v0[t].z, a0.z); a0.w = fmaf(wj[t], v0[t].w, a0.w);
              a1.x = fmaf(wj[t], v1[t].x, a1.x); a1.y = fmaf(wj[t], v1[t].y, a1.y);
              a1.z = fmaf(wj[t], v1[t].z, a1.z); a1.w = fmaf(wj[t], v1[t].w, a1.w);
            }
          }
        }
      }
    }
    const int c0 = 4 * lane;
    tile[c0 + 0][qi] = a0.x; tile[c0 + 1][qi] = a0.y; tile[c0 + 2][qi] = a0.z; tile[c0 + 3][qi] = a0.w;
    tile[128 + c0 + 0][qi] = a1.x; tile[128 + c0 + 1][qi] = a1.y; tile[128 + c0 + 2][qi] = a1.z; tile[128 + c0 + 3][qi] = a1.w;
  }
  __syncthreads();
  // channel-major store: out[b][k][c][q0 + lane]
  for (int c = warp; c < 256; c += 8) {
    const long long q = q0 + lane;
    if (q < p.Q) p.out[(((long long)b * p.K + k) * 256 + c) * p.Q + q] = tile[c][lane];
  }
}

__global__ void usage_commit_kernel(float* use, long long ubs, float* life, long long lbs,
                                    const unsigned long long* acc, long long abs_, long long off, long long n) {
  const int b = blockIdx.y;
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) {
    const double inc = (double)acc[(long long)b * abs_ + off + i] * (1.0 / (double)(1ull << CUTIE_B200_USAGE_FRAC_BITS));
    use[(long long)b * ubs + i] += (float)inc;
    life[(long long)b * lbs + i] += 1.f;
  }
}

static int pick_splits(long long B, long long Q, long long count) {
  const long long qtiles = (Q + TQ - 1) / TQ;
  const long long ntiles = (count + TK - 1) / TK;
  long long s = num_sms() / (qtiles * B);
  if (s < 1) s = 1;
  if (s > ntiles) s = ntiles;
  if (s < 1) s = 1;
  return (int)s;
}

// ---- plan: which passes run for a bank of n_total tokens ------------------------------------------------
// exact  (0): n_total < tc_min or n_total < 2 top_k, or a call without key images: exact fp32 scan of everything
//             (affinity_scan_kernel + topk_merge_kernel)
// filter (1): the FP16 plan over the key images (affinity_f16.cu): threshold sample pass, threshold select, candidate
//             filter over the whole bank, exact re-rank of the survivors
constexpr int CAND_CAP = 16384;        // candidate slots per query (overflow => exhaustive rescan of that query)

static long long g_tc_min_override = -1;
static long long g_image_level_launches = 0;     // filter passes served from a key image (tests / diagnostics)

static long long tc_min_tokens() { return g_tc_min_override >= 0 ? g_tc_min_override : 6144; }

static bool filter_plan(long long n_total, int top_k) {
  return n_total >= tc_min_tokens() && n_total >= 2 * (long long)top_k;
}

struct WsLayout {
  size_t part, cand_idx, cand_e, count, emax;   // byte offsets
  size_t total;
};

// Every call can take the exact scan (a call without key images always does); banks that qualify for the filter plan
// also get its buffers.
static WsLayout ws_layout(long long B, long long Q, long long n_total, int top_k) {
  const int kpad = top_k <= 32 ? 32 : 64;
  WsLayout w;
  memset(&w, 0, sizeof(w));
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off += (bytes + 255) / 256 * 256; return o; };
  w.part = take((size_t)B * pick_splits(B, Q, n_total) * Q * kpad * 8);
  if (filter_plan(n_total, top_k)) {
    w.cand_idx = take((size_t)B * Q * CAND_CAP * 4);
    w.cand_e = take((size_t)B * Q * CAND_CAP * 4);
    w.count = take((size_t)B * Q * 4);
    w.emax = take((size_t)B * Q * 4);
  }
  w.total = off + 256;
  return w;
}

static int run_exact(const ScanParams& base, long long B, int nsplit, int* out_idx, float* out_w, float* out_sim,
                     unsigned long long* usage_acc, cudaStream_t st) {
  ScanParams sp = base;
  const long long ntiles = (sp.n_total + TK - 1) / TK;
  sp.nsplit = nsplit;
  sp.tiles_per_split = (int)((ntiles + nsplit - 1) / nsplit);
  if ((long long)sp.tiles_per_split * TK >= (1ll << 24)) return fail(-1, "%s: split too long", "run_exact");
  dim3 grid((unsigned)((sp.Q + TQ - 1) / TQ), (unsigned)nsplit, (unsigned)B);
  const size_t smem = sizeof(ScanSmem);
  static bool attr_done[64] = {};
  if (first_use_on_device(attr_done)) {
    cudaFuncSetAttribute(affinity_scan_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    cudaFuncSetAttribute(affinity_scan_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  }
  if (sp.kpad == 32)
    affinity_scan_kernel<1><<<grid, NT, smem, st>>>(sp);
  else
    affinity_scan_kernel<2><<<grid, NT, smem, st>>>(sp);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return set_cuda_error("affinity_scan_kernel", e);
  MergeParams mp;
  mp.part_val = sp.part_val;
  mp.part_idx = sp.part_idx;
  mp.Q = sp.Q;
  mp.n_total = sp.n_total;
  mp.nsplit = nsplit;
  mp.top_k = sp.top_k;
  mp.kpad = sp.kpad;
  mp.out_idx = out_idx;
  mp.out_w = out_w;
  mp.out_sim = out_sim;
  mp.usage_acc = usage_acc;
  dim3 mgrid((unsigned)((sp.Q + 7) / 8), (unsigned)B);
  if (sp.kpad == 32)
    topk_merge_kernel<1><<<mgrid, 256, 0, st>>>(mp);
  else
    topk_merge_kernel<2><<<mgrid, 256, 0, st>>>(mp);
  e = cudaGetLastError();
  if (e != cudaSuccess) return set_cuda_error("topk_merge_kernel", e);
  return 0;
}

// Optional per-phase timing of the filtered plan (diagnostics: bench.py --phase-timing).  Events are recorded on
// the caller's stream, so they measure the kernels in situ; nothing synchronises until the times are read.
constexpr int PH_RING = 64, PH_MAX = 16;
static bool g_phase_on = false;
static cudaEvent_t g_phase_ev[PH_RING][PH_MAX];
static int g_phase_n[PH_RING];
static long long g_phase_calls = 0;
static bool g_phase_init = false;

static void phase_mark(int slot, cudaStream_t st) {
  if (!g_phase_on || slot < 0) return;
  if (g_phase_n[slot] < PH_MAX) cudaEventRecord(g_phase_ev[slot][g_phase_n[slot]++], st);
}
static int phase_begin(cudaStream_t st) {
  if (!g_phase_on) return -1;
  if (!g_phase_init) {
    for (int i = 0; i < PH_RING; ++i)
      for (int j = 0; j < PH_MAX; ++j) cudaEventCreate(&g_phase_ev[i][j]);
    g_phase_init = true;
  }
  const int slot = (int)(g_phase_calls++ % PH_RING);
  g_phase_n[slot] = 0;
  phase_mark(slot, st);
  return slot;
}

// Precomputed operand images of the arenas the segments live in (cutie_bank_key_image).
struct ImageArgs {
  const float* mu;            // [B][64] key centre of the images (null = 0)
  const int* seed_idx;        // [B][Q][kpad] threshold seeds (null = none)
  const float* img[kMaxSeg];
  long long bs[kMaxSeg];      // batch stride (floats)
  long long phys[kMaxSeg];    // physical index of the segment's first token inside its arena
};

// FP16 plan over the key operand image: tile-sampled threshold pass -> k-th smallest slot minimum -> candidate filter
// over the whole image -> exact re-rank.  Two memsets + four launches per call, whatever the bank size.
static int run_filtered_f16(const ScanParams& base, long long B, char* ws, const WsLayout& wl, int* out_idx, float* out_w,
                            float* out_sim, unsigned long long* usage_acc, const ImageArgs& ia, cudaStream_t st) {
  F16FilterParams fp;
  memset(&fp, 0, sizeof(fp));
  fp.segs = base.segs;
  fp.qk = base.qk;
  fp.qe = base.qe;
  fp.key_mu = ia.mu;
  fp.Q = base.Q;
  long long cum = 0;
  for (int s = 0; s < base.segs.nseg; ++s) {
    const long long n = base.segs.begin[s + 1] - base.segs.begin[s];
    fp.img[s] = reinterpret_cast<const unsigned char*>(ia.img[s]);
    fp.img_bs[s] = ia.bs[s] * 4;
    fp.img_tile0[s] = ia.phys[s] / 128;
    fp.img_lo0[s] = (int)(ia.phys[s] % 128);
    fp.img_tcum[s] = cum;
    cum += n > 0 ? (fp.img_lo0[s] + n + 127) / 128 : 0;
  }
  for (int s = base.segs.nseg; s <= kMaxSeg; ++s) fp.img_tcum[s] = cum;
  const int grid_x = f16_schedule(fp, B);
  const int groups = (fp.full_groups > 0 ? fp.splits_full : fp.splits_half) * 2 * F16_SLOTS;    // threshold slots per query
  if (groups > CAND_CAP) return fail(-1, "%s: too many key splits for the threshold workspace", "run_filtered_f16");
  // sample every `stride`-th tile: every split of a query group should still see >= 8 tiles (its 64 slots then hold
  // minima over >= 16 tokens each); small banks are sampled whole
  const long long max_splits = fp.full_groups > 0 ? fp.splits_full : fp.splits_half;
  long long stride = cum / (8ll * max_splits);
  if (stride > 8) stride = 8;
  if (stride < 1) stride = 1;
  const int ph = phase_begin(st);
  float* group_min = (float*)(ws + wl.cand_e);
  float* emax = (float*)(ws + wl.emax);
  cudaError_t e = cudaMemsetAsync(group_min, 0x7f, (size_t)B * base.Q * groups * 4, st);      // 0x7f7f7f7f = 3.4e38: "empty slot"
  if (e != cudaSuccess) return set_cuda_error("cudaMemsetAsync", e);
  fp.tile_stride = (int)stride;
  fp.tile_phase = 0;
  fp.group_min = group_min;
  fp.groups_per_query = groups;
  int rc = launch_f16_filter(fp, B, grid_x, true, st);
  if (rc) return rc;
  phase_mark(ph, st);
  F16ThresholdParams tp;
  memset(&tp, 0, sizeof(tp));
  tp.group_min = group_min;
  tp.groups = groups;
  tp.top_k = base.top_k;
  tp.kpad = base.kpad;
  tp.Q = base.Q;
  tp.n_total = base.n_total;
  tp.emax_out = emax;
  tp.seed_idx = ia.seed_idx;
  tp.segs = base.segs;
  tp.qk = base.qk;
  tp.qe = base.qe;
  rc = launch_f16_threshold(tp, B, st);
  if (rc) return rc;
  phase_mark(ph, st);
  e = cudaMemsetAsync(ws + wl.count, 0, (size_t)B * base.Q * 4, st);
  if (e != cudaSuccess) return set_cuda_error("cudaMemsetAsync", e);
  fp.emax_in = emax;
  fp.cand_idx = (int*)(ws + wl.cand_idx);
  fp.count = (int*)(ws + wl.count);
  fp.cap = CAND_CAP;
  rc = launch_f16_filter(fp, B, grid_x, false, st);
  if (rc) return rc;
  ++g_image_level_launches;
  phase_mark(ph, st);
  RerankParams rp;
  memset(&rp, 0, sizeof(rp));
  rp.segs = base.segs;
  rp.qk = base.qk;
  rp.qe = base.qe;
  rp.Q = base.Q;
  rp.n_total = base.n_total;
  rp.cand_idx = (const int*)(ws + wl.cand_idx);
  rp.count = (const int*)(ws + wl.count);
  rp.cap = CAND_CAP;
  rp.top_k = base.top_k;
  rp.kpad = base.kpad;
  rp.out_idx = out_idx;
  rp.out_w = out_w;
  rp.out_sim = out_sim;
  rp.usage_acc = usage_acc;
  rc = launch_rerank(rp, B, st);
  phase_mark(ph, st);
  return rc;
}

}  // namespace cutie

using namespace cutie;

extern "C" int cutie_b200_abi_version(void) { return CUTIE_B200_ABI_VERSION; }
extern "C" const char* cutie_b200_last_error(void) { return g_last_error; }

extern "C" size_t cutie_affinity_workspace_bytes(int64_t B, int64_t Q, int64_t n_total, int top_k) {
  return ws_layout(B, Q, n_total, top_k).total;
}

// Banks with fewer tokens than this use the exact scan only (default 6144).  Negative restores the default.
// Process-wide; meant for tests and tuning.
extern "C" void cutie_set_tc_min_tokens(int64_t n) { g_tc_min_override = n; }

// Per-phase device times (ms) of a filtered cutie_affinity_topk call: sample pass, threshold select, filter pass, re-rank.
// cutie_debug_phase_timing(1) starts recording (a ring of the last 64 calls); cutie_debug_phase_times(calls_ago, ...)
// waits for that call's last event and returns the number of phases written.
extern "C" void cutie_debug_phase_timing(int enable) { g_phase_on = enable != 0; }
extern "C" int cutie_debug_phase_times(int64_t calls_ago, float* out_ms, int max_phases) {
  if (!g_phase_init || calls_ago < 0 || calls_ago >= PH_RING || calls_ago >= g_phase_calls || !out_ms) return 0;
  const int slot = (int)((g_phase_calls - 1 - calls_ago) % PH_RING);
  const int n = g_phase_n[slot];
  if (n < 2) return 0;
  if (cudaEventSynchronize(g_phase_ev[slot][n - 1]) != cudaSuccess) return 0;
  int k = 0;
  for (int i = 1; i < n && k < max_phases; ++i, ++k)
    if (cudaEventElapsedTime(&out_ms[k], g_phase_ev[slot][i - 1], g_phase_ev[slot][i]) != cudaSuccess) return k;
  return k;
}

// How many filter passes have been served from a key image so far in this process (diagnostics / tests).
extern "C" int64_t cutie_debug_image_level_launches(void) { return g_image_level_launches; }

// Which plan cutie_affinity_topk_img will use when every segment has a key image: 0 = exact scan, 1 = FP16 filter.
extern "C" int cutie_affinity_plan(int64_t n_total, int top_k) { return filter_plan(n_total, top_k) ? 1 : 0; }

// Diagnostics: byte offset of the per-query candidate counters [B][Q] int32 inside the workspace (-1: exact-scan plan).
extern "C" int64_t cutie_debug_ws_count_offset(int64_t B, int64_t Q, int64_t n_total, int top_k) {
  if (!filter_plan(n_total, top_k)) return -1;
  return (int64_t)ws_layout(B, Q, n_total, top_k).count;
}

static int fill_scan_params(ScanParams& sp, int num_segments, const void* const* seg_key,
                            const void* const* seg_shrinkage, const int64_t* seg_len,
                            const int64_t* seg_key_bstride, const int64_t* seg_shr_bstride, const float* qk,
                            const float* qe, int64_t Q, int top_k, int kpad, int64_t n_total) {
  memset(&sp, 0, sizeof(sp));
  long long tot = 0;
  for (int s = 0; s < num_segments; ++s) {
    if (seg_len[s] < 0) return fail(-1, "%s: negative segment length", "cutie_affinity_topk");
    sp.segs.key[s] = (const float*)seg_key[s];
    sp.segs.shr[s] = (const float*)seg_shrinkage[s];
    sp.segs.key_bs[s] = seg_key_bstride[s];
    sp.segs.shr_bs[s] = seg_shr_bstride[s];
    sp.segs.begin[s] = tot;
    tot += seg_len[s];
  }
  for (int s = num_segments; s <= kMaxSeg; ++s) sp.segs.begin[s] = tot;
  sp.segs.nseg = num_segments;
  if (tot != n_total) return fail(-1, "%s: n_total != sum of segment lengths", "cutie_affinity_topk");
  sp.qk = qk;
  sp.qe = qe;
  sp.Q = Q;
  sp.n_total = n_total;
  sp.top_k = top_k;
  sp.kpad = kpad;
  return 0;
}

extern "C" int cutie_affinity_topk_img(int num_segments, const void* const* seg_key,
                                       const void* const* seg_shrinkage, const int64_t* seg_len,
                                       const int64_t* seg_key_bstride, const int64_t* seg_shr_bstride,
                                       const void* const* seg_key_image, const int64_t* seg_image_bstride,
                                       const int64_t* seg_phys_begin, const float* key_mu, const int32_t* seed_idx,
                                       const float* qk, const float* qe, int64_t B,
                                       int64_t CK, int64_t Q, int top_k, int kpad, int32_t* out_idx, float* out_w,
                                       float* out_sim, unsigned long long* usage_acc, int64_t n_total,
                                       void* workspace, size_t workspace_bytes, void* stream) {
  CUTIE_REQUIRE(num_segments >= 1 && num_segments <= kMaxSeg, "1..4 segments");
  CUTIE_REQUIRE(CK == CKD, "CK must be 64");
  CUTIE_REQUIRE(kpad == 32 || kpad == 64, "kpad must be 32 or 64");
  CUTIE_REQUIRE(top_k >= 1 && top_k <= kpad, "1 <= top_k <= kpad");
  CUTIE_REQUIRE(B >= 1 && Q >= 1 && qk && qe && out_idx && out_w && workspace, "null/empty argument");
  CUTIE_REQUIRE(n_total >= top_k, "selected index k out of range (top_k > number of memory tokens)");
  CUTIE_REQUIRE(n_total < (1ll << 31), "bank too large for int32 indices");
  ScanParams sp;
  int rc = fill_scan_params(sp, num_segments, seg_key, seg_shrinkage, seg_len, seg_key_bstride, seg_shr_bstride, qk,
                            qe, Q, top_k, kpad, n_total);
  if (rc) return rc;
  const WsLayout wl = ws_layout(B, Q, n_total, top_k);
  CUTIE_REQUIRE(workspace_bytes >= wl.total, "workspace too small");
  char* ws = (char*)workspace;
  cudaStream_t st = (cudaStream_t)stream;
  if (filter_plan(n_total, top_k) && seg_key_image) {
    CUTIE_REQUIRE(seg_image_bstride && seg_phys_begin, "image strides / physical offsets missing");
    ImageArgs ia;
    memset(&ia, 0, sizeof(ia));
    ia.mu = key_mu;
    ia.seed_idx = seed_idx;
    bool all_images = true;
    for (int s = 0; s < num_segments; ++s) {
      if (seg_len[s] > 0 && !seg_key_image[s]) all_images = false;     // a segment without an image: exact scan
      CUTIE_REQUIRE(seg_phys_begin[s] >= 0, "negative physical offset");
      CUTIE_REQUIRE(((uintptr_t)seg_key_image[s] & 15) == 0, "key image must be 16-byte aligned");
      ia.img[s] = (const float*)seg_key_image[s];
      ia.bs[s] = seg_image_bstride[s];
      ia.phys[s] = seg_phys_begin[s];
    }
    if (all_images) return run_filtered_f16(sp, B, ws, wl, out_idx, out_w, out_sim, usage_acc, ia, st);
  }
  const int ns0 = pick_splits(B, Q, n_total);
  sp.part_val = (float*)(ws + wl.part);
  sp.part_idx = (int*)(ws + wl.part + (size_t)B * ns0 * Q * kpad * 4);
  return run_exact(sp, B, ns0, out_idx, out_w, out_sim, usage_acc, st);
}

extern "C" int cutie_affinity_topk(int num_segments, const void* const* seg_key, const void* const* seg_shrinkage,
                                   const int64_t* seg_len, const int64_t* seg_key_bstride,
                                   const int64_t* seg_shr_bstride, const float* qk, const float* qe, int64_t B,
                                   int64_t CK, int64_t Q, int top_k, int kpad, int32_t* out_idx, float* out_w,
                                   float* out_sim, unsigned long long* usage_acc, int64_t n_total, void* workspace,
                                   size_t workspace_bytes, void* stream) {
  return cutie_affinity_topk_img(num_segments, seg_key, seg_shrinkage, seg_len, seg_key_bstride, seg_shr_bstride,
                                 nullptr, nullptr, nullptr, nullptr, nullptr, qk, qe, B, CK, Q, top_k, kpad, out_idx, out_w,
                                 out_sim,
                                 usage_acc, n_total, workspace, workspace_bytes, stream);
}

extern "C" int cutie_topk_merge(const float* part_val, const int32_t* part_idx, int64_t B, int64_t nparts, int64_t Q,
                                int top_k, int kpad, int32_t* out_idx, float* out_w, float* out_sim,
                                unsigned long long* usage_acc, int64_t n_total, void* stream) {
  CUTIE_REQUIRE(part_val && part_idx && out_idx && out_w, "null argument");
  CUTIE_REQUIRE(kpad == 32 || kpad == 64, "kpad must be 32 or 64");
  CUTIE_REQUIRE(top_k >= 1 && top_k <= kpad && nparts >= 1 && B >= 1 && Q >= 1, "bad sizes");
  MergeParams mp;
  mp.part_val = part_val;
  mp.part_idx = part_idx;
  mp.Q = Q;
  mp.n_total = n_total;
  mp.nsplit = (int)nparts;
  mp.top_k = top_k;
  mp.kpad = kpad;
  mp.out_idx = out_idx;
  mp.out_w = out_w;
  mp.out_sim = out_sim;
  mp.usage_acc = usage_acc;
  dim3 mgrid((unsigned)((Q + 7) / 8), (unsigned)B);
  if (kpad == 32)
    topk_merge_kernel<1><<<mgrid, 256, 0, (cudaStream_t)stream>>>(mp);
  else
    topk_merge_kernel<2><<<mgrid, 256, 0, (cudaStream_t)stream>>>(mp);
  CUTIE_CHECK_LAUNCH();
  return 0;
}

extern "C" int cutie_readout_gather(const int32_t* idx, const float* w, int64_t B, int64_t Q, int kpad,
                                    int num_segments, const int64_t* seg_len, const void* const* seg_val,
                                    const int64_t* seg_val_bstride, int64_t K, int64_t CV, float* out, void* stream) {
  CUTIE_REQUIRE(num_segments >= 1 && num_segments <= kMaxSeg, "1..4 segments");
  CUTIE_REQUIRE(CV == 256, "CV must be 256");
  CUTIE_REQUIRE(K >= 1 && K <= 16, "1..16 objects per call");
  CUTIE_REQUIRE(kpad == 32 || kpad == 64, "kpad must be 32 or 64");
  CUTIE_REQUIRE(idx && w && out, "null argument");
  GatherParams gp;
  memset(&gp, 0, sizeof(gp));
  long long tot = 0;
  for (int s = 0; s < num_segments; ++s) {
    gp.segs.begin[s] = tot;
    tot += seg_len[s];
    for (int k = 0; k < K; ++k) {
      gp.segs.rows[s * K + k] = (const float*)seg_val[s * K + k];
      gp.segs.bs[s * K + k] = seg_val_bstride[s * K + k];
    }
  }
  for (int s = num_segments; s <= kMaxSeg; ++s) gp.segs.begin[s] = tot;
  gp.segs.nseg = num_segments;
  gp.segs.nobj = (int)K;
  gp.idx = idx;
  gp.w = w;
  gp.Q = Q;
  gp.kpad = kpad;
  gp.K = K;
  gp.CV = CV;
  gp.out = out;
  dim3 grid((unsigned)((Q + GQ - 1) / GQ), (unsigned)K, (unsigned)B);
  readout_gather_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(gp);
  CUTIE_CHECK_LAUNCH();
  return 0;
}

extern "C" int cutie_usage_commit(float* use_cnt, int64_t use_bstride, float* life_cnt, int64_t life_bstride,
                                  const unsigned long long* usage_acc, int64_t acc_bstride, int64_t acc_offset,
                                  int64_t B, int64_t n, void* stream) {
  CUTIE_REQUIRE(use_cnt && life_cnt && usage_acc, "null argument");
  if (n <= 0) return 0;
  dim3 grid((unsigned)((n + 255) / 256), (unsigned)B);
  usage_commit_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(use_cnt, use_bstride, life_cnt, life_bstride, usage_acc,
                                                             acc_bstride, acc_offset, n);
  CUTIE_CHECK_LAUNCH();
  return 0;
}
