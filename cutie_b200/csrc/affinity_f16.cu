// FP16 tcgen05 candidate filter over the memory bank's key operand image (sm_100a) -- the large-bank plan of
// cutie_affinity_topk (get_similarity + top-k of do_softmax, cutie/model/utils/memory_utils.py:7-77).
//
//   E[q,n] = -8 S[q,n] = shr_n sum_c qe_c (k_c - qk_c)^2 = [qe | -2 qe qk | tail] . [shr k^2 | shr k | tail]    (K = 128 + 16)
//
// Both operands are K-major FP16 (tc_operand_f16.cuh); the key side is the bank's precomputed image, fetched with ONE
// 36 KB bulk copy per 128-token tile (3 stages); the query side is built once per CTA for 256 queries (two M = 128
// halves: every key tile is multiplied by both, which halves the L2 -> SM bytes per flop again).  kind::f16 MMAs with
// fp32 accumulators double-buffered in TMEM (2 x 2 x 128 columns = all 512).
//
// The tail columns make the MMA itself emit a rigorous bound of the exact energy:
//   filter pass  (sign +1): D = E_f16 - eps (P_n + R_n v_q)^2 - abs  <=  E_exact        -> candidate iff D < Emax_q
//   sample pass  (sign -1): U = E_f16 + eps (P_n + R_n v_q)^2 + abs  >=  E_exact        -> threshold seeding
// so a true top-k member is never dropped; survivors are re-ranked with the exact fp32 direct form
// (affinity_rerank_kernel, below), which makes the final selection and weights bit-identical to the exact scan.
//
// Threshold seeding without a select over a token list: the sample pass walks every `stride`-th tile of the image and
// every epilogue thread (= one query x one 64-column group of one CTA) keeps 32 running minima of U, one per register
// of its tcgen05.ld -- 1 FMNMX per element, no memory traffic.  The minima of different (CTA, column group, register)
// slots belong to DISJOINT token sets, so the k-th smallest of a query's slot minima is an upper bound of its k-th
// smallest exact energy (f16_threshold_kernel).  8 slots per thread (register j folds into slot j % 8): with 22 key
// splits a query owns 352 disjoint groups -- ~1.3 expected collisions among its 30 best, i.e. the bound lands on the
// ~31st smallest instead of the 30th -- and the threshold kernel handles 11 values per lane instead of 44.
//
// Warp roles (576 threads): warps 0-15 epilogue (TMEM lane quarter = w & 3, query half = (w >> 2) & 1, 64-column group
// = w >> 3), warp 16 bulk-copy producer (one thread), warp 17 TMEM allocator + single-thread MMA issuer.
#include "topk_common.cuh"
#include "affinity_internal.cuh"
#include "tc_operand_f16.cuh"
#include "tc_ptx.cuh"

namespace cutie {

namespace {

constexpr int F16_THREADS = 576;
constexpr int F16_STAGES = 3;
constexpr int F16_QT = 256;                 // queries per CTA (two MMA M = 128 halves)

struct F16Tail {
  unsigned long long full[F16_STAGES], empty[F16_STAGES], tfull[2], tempty[2], aready;
  uint32_t tmem_base;
  float thr[F16_QT];          // per query row: filter threshold (filter pass) / +inf for a query that cannot be bounded (sample pass)
};

struct F16Tile {
  const unsigned char* src;   // F16_OPER_BYTES contiguous bytes: the tile exactly as the MMA wants it in shared memory
  int lo, hi;                 // rows [lo, hi) of the tile belong to the segment
  long long lbase;            // bank (logical) index of row 0
};
__device__ __forceinline__ F16Tile f16_tile(const F16FilterParams& p, int b, long long g) {
  int s = 0;
#pragma unroll
  for (int i = 1; i < kMaxSeg; ++i)
    if (i < p.segs.nseg && g >= p.img_tcum[i]) s = i;
  const long long j = g - p.img_tcum[s];
  const long long n = p.segs.begin[s + 1] - p.segs.begin[s];
  const long long lo0 = p.img_lo0[s];
  const long long a = lo0 - j * F16_KTILE, e = lo0 + n - j * F16_KTILE;
  F16Tile t;
  t.lo = a < 0 ? 0 : (int)a;
  t.hi = e > F16_KTILE ? F16_KTILE : (int)e;
  t.lbase = p.segs.begin[s] - lo0 + j * F16_KTILE;
  t.src = p.img[s] + (long long)b * p.img_bs[s] + (p.img_tile0[s] + j) * (long long)F16_OPER_BYTES;
  return t;
}
__device__ __forceinline__ unsigned range_mask32(int a, int b) {      // bits [a, b) of a 32-bit word (any ints)
  const unsigned hi = b >= 32 ? 0xffffffffu : (b <= 0 ? 0u : ((1u << b) - 1u));
  const unsigned lo = a <= 0 ? 0xffffffffu : (a >= 32 ? 0u : ~((1u << a) - 1u));
  return hi & lo;
}
// three-input minimum (sm_100+): one ALU-pipe instruction per two new elements.  The epilogue is bound by the ALU pipe
// (one warp instruction per 2 cycles per scheduler: ncu "math pipe throttle" was the top stall of the compare-and-mask
// formulation, 2+ instructions per accumulator element), so everything per-element goes through min3 trees.
__device__ __forceinline__ float fmin3(float a, float b, float c) {
  float d;
  asm("min.f32 %0, %1, %2, %3;" : "=f"(d) : "f"(a), "f"(b), "f"(c));
  return d;
}
__device__ __forceinline__ float min32(const uint32_t (&r)[32]) {
  float m[11];
#pragma unroll
  for (int i = 0; i < 10; ++i) m[i] = fmin3(__uint_as_float(r[3 * i]), __uint_as_float(r[3 * i + 1]), __uint_as_float(r[3 * i + 2]));
  m[10] = fminf(__uint_as_float(r[30]), __uint_as_float(r[31]));
  const float a = fmin3(m[0], m[1], m[2]), b = fmin3(m[3], m[4], m[5]), c = fmin3(m[6], m[7], m[8]);
  return fmin3(fmin3(a, b, c), m[9], m[10]);
}
// K-major un-swizzled (interleaved 8 x 16 B core matrices) descriptor of the [128 x 32 B] tail block
__device__ __forceinline__ uint64_t desc_tail16(uint32_t addr) {
  uint64_t d = 0;
  d |= (uint64_t)((addr >> 4) & 0x3FFF);
  d |= (uint64_t)(2048 >> 4) << 16;              // LBO: distance between the two 16-B K chunks
  d |= (uint64_t)(128 >> 4) << 32;               // SBO: distance between 8-row groups
  d |= (uint64_t)1 << 46;
  return d;
}

}  // namespace

template <bool SAMPLE>
__global__ void __launch_bounds__(F16_THREADS, 1) affinity_f16_filter_kernel(const F16FilterParams p) {
  extern __shared__ __align__(1024) unsigned char smem[];
  unsigned char* A = smem;                                   // 2 query halves
  unsigned char* Bst = smem + 2 * F16_OPER_BYTES;            // F16_STAGES key tiles
  F16Tail& T = *reinterpret_cast<F16Tail*>(smem + (2 + F16_STAGES) * F16_OPER_BYTES);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int b = blockIdx.y;
  // CTA -> (query group, key split): full groups (256 queries) get `splits_full` CTAs each, a trailing group with at
  // most 128 queries gets `splits_half` (half the MMA work per tile)
  int grp, split, nsplit;
  {
    const int bid = blockIdx.x, nf = p.full_groups * p.splits_full;
    if (bid < nf) { grp = bid / p.splits_full; split = bid % p.splits_full; nsplit = p.splits_full; }
    else { grp = p.full_groups; split = bid - nf; nsplit = p.splits_half; }
  }
  const long long q0 = (long long)grp * F16_QT;
  const int halves = (q0 + 128 < p.Q) ? 2 : 1;
  // tiles of this CTA: physical image tiles g (SAMPLE: only g = phase + j * stride), dealt round-robin to the splits
  const long long all_tiles = p.img_tcum[p.segs.nseg];
  const long long my_pool = SAMPLE ? (all_tiles > p.tile_phase ? (all_tiles - p.tile_phase + p.tile_stride - 1) / p.tile_stride : 0)
                                   : all_tiles;
  const int ntiles = split < my_pool ? (int)((my_pool - split + nsplit - 1) / nsplit) : 0;
  auto tile_of = [&](int t) -> long long {
    const long long j = (long long)split + (long long)t * nsplit;
    return SAMPLE ? (long long)p.tile_phase + j * p.tile_stride : j;
  };

  if (tid == 0) {
    for (int s = 0; s < F16_STAGES; ++s) { mbar_init(smem_u32(&T.full[s]), 1); mbar_init(smem_u32(&T.empty[s]), 1); }
    for (int a = 0; a < 2; ++a) { mbar_init(smem_u32(&T.tfull[a]), 1); mbar_init(smem_u32(&T.tempty[a]), 32 * 8 * halves); }
    mbar_init(smem_u32(&T.aready), F16_QT);
    mbar_init_fence();
  }
  if (warp == 17) tmem_alloc<512>(smem_u32(&T.tmem_base));
  tc_fence_before();
  __syncthreads();          // barriers + TMEM exist; from here the roles run free: the key tiles are already being copied
  tc_fence_after();         // while warps 0-7 build the query operand (the MMA issuer waits for `aready`)
  const uint32_t tmem = T.tmem_base;
  // ---- query operand: thread == query row (tid < 256): [qe | -2 qe qk] + tail ----
  if (tid < F16_QT) {
    const int half = tid >> 7, row = tid & 127;
    unsigned char* Ah = A + half * F16_OPER_BYTES;
    const long long q = q0 + tid;
    const bool qok = q < p.Q;
    const float* qe_p = p.qe + (long long)b * CKD * p.Q + (qok ? q : 0);
    const float* qk_p = p.qk + (long long)b * CKD * p.Q + (qok ? q : 0);
    float b2 = 0.f, a1 = 0.f;
    // 32 channels per batch: 64 independent loads in flight (the prologue is latency-bound and sits on every CTA's path)
#pragma unroll 1
    for (int cb = 0; cb < CKD; cb += 32) {
      float ev[32], kv[32];
#pragma unroll
      for (int i = 0; i < 32; ++i) {
        ev[i] = qok ? __ldg(qe_p + (long long)(cb + i) * p.Q) : 0.f;
        kv[i] = qok ? __ldg(qk_p + (long long)(cb + i) * p.Q) - (p.key_mu ? __ldg(p.key_mu + b * CKD + cb + i) : 0.f) : 0.f;
      }
#pragma unroll
      for (int g8 = 0; g8 < 4; ++g8) {
        uint32_t w0[4], w1[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const float e0 = ev[8 * g8 + 2 * i], e1 = ev[8 * g8 + 2 * i + 1], k0 = kv[8 * g8 + 2 * i], k1 = kv[8 * g8 + 2 * i + 1];
          b2 = fmaf(e0 * k0, k0, b2);
          b2 = fmaf(e1 * k1, k1, b2);
          a1 += e0 + 2.f * e0 * fabsf(k0) + e1 + 2.f * e1 * fabsf(k1);
          w0[i] = pack_rn(e0, e1);
          w1[i] = pack_rn(-2.f * e0 * k0, -2.f * e1 * k1);
        }
        *reinterpret_cast<uint4*>(Ah + f16_off_main(row, cb + 8 * g8)) = make_uint4(w0[0], w0[1], w0[2], w0[3]);
        *reinterpret_cast<uint4*>(Ah + f16_off_main(row, 64 + cb + 8 * g8)) = make_uint4(w1[0], w1[1], w1[2], w1[3]);
      }
    }
    // tail: [b2_hi, b2_lo, s, s v, s v^2, s, -s absA, s | 0 x 8] with s = +1 (filter: lower bound) / -1 (sample: upper)
    const bool fits = qok && b2 <= 3.0e4f;            // v^2 must fit f16; otherwise the query is not filtered at all
    const float sgn = SAMPLE ? -1.f : 1.f;
    const __half b2h = __float2half_rn(fits ? b2 : 0.f);
    const __half b2l = __float2half_rn(fits ? b2 - __half2float(b2h) : 0.f);
    const float v = fits ? sqrtf(b2) * 1.001f : 0.f;
    const float absa = F16_ABS * (a1 + b2 + v + v * v + 8.f);
    uint4 t0, t1 = make_uint4(0u, 0u, 0u, 0u);
    t0.x = pack_h2(b2h, b2l);
    t0.y = pack_h2(__float2half_rn(sgn), h_up(sgn * v));
    t0.z = pack_h2(h_up(sgn * v * v * 1.001f), __float2half_rn(sgn));
    t0.w = pack_h2(h_up(-sgn * absa), __float2half_rn(sgn));
    *reinterpret_cast<uint4*>(Ah + f16_off_tail(row, 0)) = t0;
    *reinterpret_cast<uint4*>(Ah + f16_off_tail(row, 8)) = t1;
    if (SAMPLE)
      T.thr[tid] = fits ? 0.f : CUDART_INF_F;
    else
      T.thr[tid] = !qok ? -CUDART_INF_F : (fits ? p.emax_in[(long long)b * p.Q + q] : CUDART_INF_F);
    fence_proxy_async();
    mbar_arrive(smem_u32(&T.aready));
  }

  if (warp < 16) {
    // =========================== epilogue: thread == (query, 64-column group) ===========================
    const int half = (warp >> 2) & 1, cg64 = warp >> 3;
    if (half < halves) {
      const long long q = q0 + half * 128 + (warp & 3) * 32 + lane;
      const bool qok = q < p.Q;
      mbar_wait(smem_u32(&T.aready), 0);                                 // the query rows (and their thresholds) exist
      const float thr = T.thr[half * 128 + (warp & 3) * 32 + lane];     // written by the thread that built this query's row
      const long long bq = (long long)b * p.Q + (qok ? q : 0);
      int* my_idx = SAMPLE ? nullptr : p.cand_idx + bq * p.cap;
      int blk_base = 0, blk_used = F16_RESERVE;
      float mn[F16_SLOTS];
      if (SAMPLE) {
#pragma unroll
        for (int j = 0; j < F16_SLOTS; ++j) mn[j] = CUDART_INF_F;
      }
      const uint32_t lane_base = tmem + ((uint32_t)((warp & 3) * 32) << 16) + (uint32_t)(half * 128 + cg64 * 64);
      for (int t = 0; t < ntiles; ++t) {
        const int a = t & 1;
        mbar_wait(smem_u32(&T.tfull[a]), (t >> 1) & 1);
        tc_fence_after();
        const F16Tile it = f16_tile(p, b, tile_of(t));
#pragma unroll 1
        for (int sub = 0; sub < 2; ++sub) {
          const int c0 = cg64 * 64 + sub * 32;
          uint32_t r[32];
          tmem_ld32(lane_base + (uint32_t)(a * 256 + sub * 32), r);
          if (SAMPLE) {
            if (it.lo <= c0 && it.hi >= c0 + 32) {
#pragma unroll
              for (int j = 0; j < F16_SLOTS; ++j) {             // 4 new values per slot: two min3
                mn[j] = fmin3(mn[j], __uint_as_float(r[j]), __uint_as_float(r[j + F16_SLOTS]));
                mn[j] = fmin3(mn[j], __uint_as_float(r[j + 2 * F16_SLOTS]), __uint_as_float(r[j + 3 * F16_SLOTS]));
              }
            } else {
              const unsigned ok = range_mask32(it.lo - c0, it.hi - c0);
#pragma unroll
              for (int j = 0; j < 32; ++j)
                mn[j % F16_SLOTS] = ((ok >> j) & 1u) ? fminf(mn[j % F16_SLOTS], __uint_as_float(r[j])) : mn[j % F16_SLOTS];
            }
          } else {
            // candidates are rare (~0.1 % of the columns): a min3 tree decides "none here" in 16 instructions; only a
            // lane that saw something builds its bitmask of passing columns and walks it
            unsigned m = 0u;
            if (min32(r) < thr) {
#pragma unroll
              for (int j = 0; j < 32; ++j) m |= (__uint_as_float(r[j]) < thr) ? (1u << j) : 0u;
              m &= range_mask32(it.lo - c0, it.hi - c0);
            }
            while (m) {
              const int j = __ffs(m) - 1;
              m &= m - 1;
              // slots are reserved in blocks: one global atomic per block of candidates of this (query, thread)
              if (blk_used == F16_RESERVE) { blk_base = atomicAdd(&p.count[bq], F16_RESERVE); blk_used = 0; }
              const int pos = blk_base + blk_used++;
              if (pos < p.cap) my_idx[pos] = (int)(it.lbase + c0 + j);
            }
            __syncwarp();      // reconverge before the next aligned tcgen05.ld / the barrier arrive
          }
        }
        tc_fence_before();
        mbar_arrive(smem_u32(&T.tempty[a]));
      }
      if (SAMPLE) {
        if (qok) {
          float* g = p.group_min + bq * (long long)p.groups_per_query + (long long)(split * 2 + cg64) * F16_SLOTS;
#pragma unroll
          for (int j = 0; j < F16_SLOTS; j += 4)      // thr = +inf marks a query whose operand row carries no valid bound
            *reinterpret_cast<float4*>(g + j) = make_float4(mn[j] + thr, mn[j + 1] + thr, mn[j + 2] + thr, mn[j + 3] + thr);
        }
      } else if (blk_used < F16_RESERVE) {
        for (int u = blk_used; u < F16_RESERVE; ++u)
          if (blk_base + u < p.cap) my_idx[blk_base + u] = -1;       // unused slots of the last block are voided
      }
    }
  } else if (warp == 16) {
    // ============ producer: one thread, one 36 KB bulk copy per tile ============
    if (lane == 0) {
      for (int t = 0; t < ntiles; ++t) {
        const int s = t % F16_STAGES;
        mbar_wait(smem_u32(&T.empty[s]), ((t / F16_STAGES) & 1) ^ 1);
        const F16Tile it = f16_tile(p, b, tile_of(t));
        const uint32_t bar = smem_u32(&T.full[s]);
        mbar_arrive_expect_tx(bar, (uint32_t)F16_OPER_BYTES);
        bulk_g2s(smem_u32(Bst + s * F16_OPER_BYTES), it.src, (uint32_t)F16_OPER_BYTES, bar);
      }
    }
  } else if (warp == 17) {
    // =========================== MMA issuer ===========================
    if (lane == 0) {
      // instruction descriptor: D = F32, A = B = F16, K-major both, N = 128, M = 128
      const uint32_t idesc = (1u << 4) | ((uint32_t)(F16_KTILE >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
      const uint32_t a_base = smem_u32(A);
      mbar_wait(smem_u32(&T.aready), 0);                       // all 256 query rows written (and proxy-fenced)
      for (int t = 0; t < ntiles; ++t) {
        const int s = t % F16_STAGES, a = t & 1;
        mbar_wait(smem_u32(&T.full[s]), (t / F16_STAGES) & 1);
        mbar_wait(smem_u32(&T.tempty[a]), ((t >> 1) & 1) ^ 1);
        tc_fence_after();
        const uint32_t b_base = smem_u32(Bst + s * F16_OPER_BYTES);
        for (int h = 0; h < halves; ++h) {
          const uint32_t d = tmem + (uint32_t)(a * 256 + h * 128);
          const uint32_t ah = a_base + h * F16_OPER_BYTES;
#pragma unroll
          for (int blk = 0; blk < 2; ++blk)
#pragma unroll
            for (int ks = 0; ks < 4; ++ks)
              tc_mma_f16(d, desc_sw128_kmajor(ah + blk * F16_BLK_BYTES + ks * 32),
                         desc_sw128_kmajor(b_base + blk * F16_BLK_BYTES + ks * 32), idesc, (blk | ks) ? 1u : 0u);
          tc_mma_f16(d, desc_tail16(ah + 2 * F16_BLK_BYTES), desc_tail16(b_base + 2 * F16_BLK_BYTES), idesc, 1u);
        }
        tc_commit(smem_u32(&T.empty[s]));
        tc_commit(smem_u32(&T.tfull[a]));
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 17) {
    tc_fence_after();
    tmem_dealloc<512>(tmem);
  }
}

// Emax[q] = k-th smallest of the query's slot minima (upper bounds of exact energies of DISJOINT token sets), one warp
// per query: the slot values live in registers (<= 64 per lane) and the k-th smallest is found by a bitwise binary search
// on the float bit patterns (energies are >= 0, so the unsigned order is the numeric order): 31 rounds of "how many values
// are <= candidate", no sorting, no shared memory, deterministic.  Fewer than k finite slots (tiny sample) => +inf: every
// token of that query is re-ranked.
constexpr int THR_PER_LANE = 16;
__global__ void __launch_bounds__(256) f16_threshold_kernel(const F16ThresholdParams p) {
  __shared__ float qab[8][2 * CKD];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const long long q = (long long)blockIdx.x * 8 + warp;
  if (q >= p.Q) return;
  const int b = blockIdx.y;
  const long long bq = (long long)b * p.Q + q;
  const float* g = p.group_min + bq * (long long)p.groups;
  uint32_t v[THR_PER_LANE];
  int finite = 0;
#pragma unroll
  for (int i = 0; i < THR_PER_LANE; ++i) {
    const int j = i * 32 + lane;
    float e = j < p.groups ? __ldg(g + j) : CUDART_INF_F;
    e = (e >= 0.f) ? e : 0.f;                                  // a bound can round a hair below zero: still an upper bound at 0+
    const bool ok = e < 1e30f;                                 // empty (memset pattern) / flagged slots never count
    v[i] = ok ? __float_as_uint(e) : 0x7f800000u;
    finite += ok ? 1 : 0;
  }
  finite = __reduce_add_sync(0xffffffffu, finite);
  float emax = CUDART_INF_F;
  if (finite >= p.top_k) {
    uint32_t prefix = 0u;                                      // bits decided so far of the k-th smallest pattern
    for (int bit = 30; bit >= 0; --bit) {
      const uint32_t cand = prefix | ((1u << bit) - 1u);       // largest pattern with this bit clear
      int c = 0;
#pragma unroll
      for (int i = 0; i < THR_PER_LANE; ++i) c += (v[i] <= cand) ? 1 : 0;
      c = __reduce_add_sync(0xffffffffu, c);
      if (c < p.top_k) prefix |= (1u << bit);                  // fewer than k values at or below: the answer has the bit set
    }
    emax = __uint_as_float(prefix) * (1.f + 1e-6f) + 1e-30f;
  }
  // Seeds: top_k DISTINCT tokens proposed by the caller (the previous frame's winners for this query position, re-indexed
  // for what the ring dropped since).  The largest of their exact energies under THIS query bounds the k-th smallest
  // exact energy -- in a temporally coherent video it is nearly the k-th smallest itself, far below what a 1/8 sample
  // can offer.  A query with an invalid seed keeps the sampled bound.
  if (p.seed_idx) {
    for (int c = lane; c < CKD; c += 32) {
      const long long off = ((long long)b * CKD + c) * p.Q + q;
      const float a = sqrtf(__ldg(p.qe + off));
      qab[warp][c] = a;
      qab[warp][CKD + c] = a * __ldg(p.qk + off);
    }
    __syncwarp();
    const bool mine = lane < p.top_k || (lane + 32 < p.top_k);
    float worst = 0.f;
    bool ok = true;
    for (int j = lane; j < p.top_k; j += 32) {
      const int id = __ldg(p.seed_idx + bq * p.kpad + j);
      const bool valid = id >= 0 && id < p.n_total;
      ok = ok && valid;
      if (valid) {
        const int sg = seg_of(p.segs.begin, p.segs.nseg, id);
        const long long off = (long long)id - p.segs.begin[sg];
        const float sv = exact_similarity(p.segs.key[sg] + (long long)b * p.segs.key_bs[sg] + off * CKD,
                                          __ldg(p.segs.shr[sg] + (long long)b * p.segs.shr_bs[sg] + off), &qab[warp][0],
                                          &qab[warp][CKD]);
        worst = fmaxf(worst, -8.f * sv);
      }
    }
    (void)mine;
    ok = __all_sync(0xffffffffu, ok);
    worst = warp_max(worst);
    if (ok) emax = fminf(emax, worst * (1.f + 1e-5f) + 1e-30f);
  }
  if (lane == 0) p.emax_out[bq] = emax;
}

// ------------------------------------------------------------------------------------------------
// Exact re-rank of the filter pass's candidates: one CTA (4 warps) per query.  Each warp evaluates chunks of 32
// candidates with the exact fp32 direct form and keeps a sorted top-k; warp 0 merges and finalises (softmax,
// usage).  A query whose candidate list overflowed is rescanned exhaustively (slow, correct, rare).
//
// Candidate key rows (256 B each) are fetched COALESCED -- a half-warp per row, 16 independent LDG.128 per lane in flight
// -- and staged in shared memory; each lane then evaluates its own candidate from shared memory with the same
// channel-sequential fp32 arithmetic as the exact scan (`exact_similarity_smem`), so results stay bit-identical.  (A lane
// reading its own row straight from global memory touches 32 different 128-byte lines per instruction: 512 L1 wavefronts
// per 32 candidates against 64 here, and the re-rank was bound by exactly that.)
constexpr int RR_LD = 68;                 // floats per staged row: 272 B, 16-byte aligned, conflict-free LDS.128 per quarter-warp

__device__ __forceinline__ float exact_similarity_smem(const float* __restrict__ krow, float shr, const float* __restrict__ a,
                                                       const float* __restrict__ b) {
  float acc = 0.f;
#pragma unroll
  for (int c4 = 0; c4 < CKD / 4; ++c4) {
    const float4 kf = *reinterpret_cast<const float4*>(krow + 4 * c4);
    float d;
    d = fmaf(a[4 * c4 + 0], kf.x, -b[4 * c4 + 0]); acc = fmaf(d, d, acc);
    d = fmaf(a[4 * c4 + 1], kf.y, -b[4 * c4 + 1]); acc = fmaf(d, d, acc);
    d = fmaf(a[4 * c4 + 2], kf.z, -b[4 * c4 + 2]); acc = fmaf(d, d, acc);
    d = fmaf(a[4 * c4 + 3], kf.w, -b[4 * c4 + 3]); acc = fmaf(d, d, acc);
  }
  return acc * (-shr * rsqrtf((float)CKD));
}

template <int NS>
__global__ void __launch_bounds__(128) affinity_rerank_kernel(const RerankParams p) {
  __shared__ float lv[4][KPAD_MAX];
  __shared__ int li[4][KPAD_MAX];
  __shared__ float qa[CKD], qb[CKD];
  __shared__ __align__(16) float rows[4][32][RR_LD];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int b = blockIdx.y;
  const long long q = blockIdx.x;
  const long long bq = (long long)b * p.Q + q;
  for (int u = 0; u < NS; ++u) { lv[warp][lane + 32 * u] = -CUDART_INF_F; li[warp][lane + 32 * u] = INT_MAX; }
  if (tid < CKD) {
    const long long off = ((long long)b * CKD + tid) * p.Q + q;
    const float a = sqrtf(p.qe[off]);
    qa[tid] = a;
    qb[tid] = a * p.qk[off];
  }
  __syncthreads();
  int n = p.count[bq];
  const bool exhaustive = n > p.cap;
  if (exhaustive) n = (int)p.n_total;
  const int* cl = p.cand_idx + bq * p.cap;
  const int h = lane >> 4, c4 = lane & 15;
  for (int base = warp * 32; base < n; base += 128) {
    const int j = base + lane;
    int id = -1;
    if (j < n) id = exhaustive ? j : cl[j];
    const bool live = id >= 0;
    float shr = 0.f;
    const float* krow = nullptr;
    if (live) {
      const int sg = seg_of(p.segs.begin, p.segs.nseg, id);
      const long long off = (long long)id - p.segs.begin[sg];
      krow = p.segs.key[sg] + (long long)b * p.segs.key_bs[sg] + off * CKD;
      shr = __ldg(p.segs.shr[sg] + (long long)b * p.segs.shr_bs[sg] + off);
    }
    // cooperative, coalesced fetch: at step it the two half-warps fetch rows 2 it and 2 it + 1 (16 lanes x 16 B each)
    float4 piece[16];
#pragma unroll
    for (int it = 0; it < 16; ++it) {
      const unsigned long long rp = __shfl_sync(0xffffffffu, (unsigned long long)krow, 2 * it + h);
      piece[it] = rp ? __ldg(reinterpret_cast<const float4*>(rp) + c4) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
#pragma unroll
    for (int it = 0; it < 16; ++it) *reinterpret_cast<float4*>(&rows[warp][2 * it + h][4 * c4]) = piece[it];
    __syncwarp();
    const float sv = live ? exact_similarity_smem(&rows[warp][lane][0], shr, qa, qb) : -CUDART_INF_F;
    if (!live) id = INT_MAX;
    const float kth = lv[warp][p.top_k - 1];
    const int kthi = li[warp][p.top_k - 1];
    unsigned bits = __ballot_sync(0xffffffffu, live && (sv > kth || (sv == kth && id < kthi)));
    while (bits) {
      const int src = __ffs(bits) - 1;
      bits &= bits - 1;
      const float cs = __shfl_sync(0xffffffffu, sv, src);
      const int ci = __shfl_sync(0xffffffffu, id, src);
      const float k2 = lv[warp][p.top_k - 1];
      if (cs > k2 || (cs == k2 && ci < li[warp][p.top_k - 1]))
        list_insert<NS>(&lv[warp][0], &li[warp][0], lane, p.top_k, cs, ci);
    }
    __syncwarp();      // the staging rows are overwritten by the next chunk
  }
  __syncthreads();
  if (warp == 0) {
    for (int w = 1; w < 4; ++w) {
      for (int j = 0; j < p.top_k; ++j) {
        const float cs = lv[w][j];
        const int ci = li[w][j];
        if (ci == INT_MAX) break;
        const float k2 = lv[0][p.top_k - 1];
        if (!(cs > k2 || (cs == k2 && ci < li[0][p.top_k - 1]))) break;     // sorted: the rest lose too
        list_insert<NS>(&lv[0][0], &li[0][0], lane, p.top_k, cs, ci);
      }
    }
    const long long oo = bq * p.kpad;
    finalize_topk<NS>(&lv[0][0], &li[0][0], lane, p.top_k, p.kpad, p.out_idx + oo, p.out_w + oo,
                      p.out_sim ? p.out_sim + oo : nullptr,
                      p.usage_acc ? p.usage_acc + (long long)b * p.n_total : nullptr);
  }
}

size_t f16_filter_smem_bytes() { return (size_t)(2 + F16_STAGES) * F16_OPER_BYTES + sizeof(F16Tail) + 64; }

// CTA schedule for Q queries: returns the grid size; fills the group / split counts of `p`
int f16_schedule(F16FilterParams& p, long long B) {
  const int sms = num_sms();
  p.full_groups = (int)(p.Q / F16_QT);
  const long long rest = p.Q - (long long)p.full_groups * F16_QT;
  int half_groups = 0;
  if (rest > 128) { ++p.full_groups; }          // a trailing group with two live halves counts as a full one
  else if (rest > 0) half_groups = 1;
  const long long units = 2ll * p.full_groups + half_groups;             // half-tile work units per key tile
  long long u = sms / (units * B);
  if (u < 1) u = 1;
  if (u > 16) u = 16;                              // 2u splits x 16 threshold slots <= 512 (f16_threshold_kernel)
  const long long tiles = p.img_tcum[p.segs.nseg];
  if (2 * u > tiles) u = (tiles + 1) / 2 > 0 ? (tiles + 1) / 2 : 1;
  p.splits_full = (int)(2 * u);
  p.splits_half = half_groups ? (int)u : 0;
  return p.full_groups * p.splits_full + p.splits_half;
}

int launch_f16_filter(const F16FilterParams& p, long long B, int grid_x, bool sample, cudaStream_t st) {
  const size_t smem = f16_filter_smem_bytes();
  static bool attr_done[64] = {};
  if (first_use_on_device(attr_done)) {
    cudaFuncSetAttribute(affinity_f16_filter_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    cudaFuncSetAttribute(affinity_f16_filter_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  }
  dim3 grid((unsigned)grid_x, (unsigned)B);
  if (sample)
    affinity_f16_filter_kernel<true><<<grid, F16_THREADS, smem, st>>>(p);
  else
    affinity_f16_filter_kernel<false><<<grid, F16_THREADS, smem, st>>>(p);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return set_cuda_error("affinity_f16_filter_kernel", e);
  return 0;
}

int launch_f16_threshold(const F16ThresholdParams& p, long long B, cudaStream_t st) {
  if (p.groups > THR_PER_LANE * 32) return fail(-1, "%s: too many threshold slots", "f16_threshold_kernel");
  dim3 grid((unsigned)((p.Q + 7) / 8), (unsigned)B);
  f16_threshold_kernel<<<grid, 256, 0, st>>>(p);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return set_cuda_error("f16_threshold_kernel", e);
  return 0;
}

int launch_rerank(const RerankParams& p, long long B, cudaStream_t st) {
  dim3 grid((unsigned)p.Q, (unsigned)B);
  if (p.kpad == 32)
    affinity_rerank_kernel<1><<<grid, 128, 0, st>>>(p);
  else
    affinity_rerank_kernel<2><<<grid, 128, 0, st>>>(p);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return set_cuda_error("affinity_rerank_kernel", e);
  return 0;
}

}  // namespace cutie
