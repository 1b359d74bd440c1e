// rp_score_topk.cu - fused predict head:  scores = Hq[B,d] . E[I,d]^T  ->  seen-item mask  ->  per-row top-K.
//
// Replaces, for one batch of users, the reference chain
//   EmbeddingTyingHead.forward            replay/nn/head.py:29-34   (legacy: models/nn/sequential/sasrec/model.py:286-307)
//   SeenItemsFilter._compute_scores       replay/nn/lightning/postprocessor/seen_items.py:56-83
//   torch.topk(logits, k, dim=1)          replay/nn/lightning/callback/predictions_callback.py:90
// without ever materialising the [B, |I|] logits.
//
// Kernel 1 (score_topk_kernel): one CTA = 128 users x a contiguous range of 128-item tiles.
//   warp 0   TMA producer: user tile A (resident in smem) + ring of item-table K-chunks [128 items x 64]
//   warp 1   tcgen05.mma issuer: S[128x128] fp32 in TMEM, double buffered (2 x 128 columns)
//   warps 2-5 epilogue: tcgen05.ld 32 columns at a time, thread = user row, seen-mask via a cursor into the user's
//            sorted seen list, running top-K (sorted, registers), partial top-K written per (user, item split)
// Kernel 2 (topk_merge_kernel): one warp per user merges the per-split partial lists (score desc, column asc).
#include "rp_host.h"
#include "rp_sm100.cuh"

namespace rp {

static constexpr int kTileM = 128;   // users per CTA
static constexpr int kTileN = 128;   // items per MMA tile
static constexpr int kChunkBytes = 128 * 128;  // [128 rows x 64 bf16]
static constexpr int kNoId = 0x7fffffff;

// Per-thread running top-K kept in registers.  The K live entries occupy slots [KMAX-K, KMAX) in descending order so
// that the admission threshold is always the statically indexed last slot; slots below hold +inf sentinels that never
// move.  (A runtime-indexed v[K-1] would push the whole structure into local memory.)
template <int KMAX>
struct TopK {
  float v[KMAX];
  int id[KMAX];
  __device__ __forceinline__ void init(int K) {
#pragma unroll
    for (int i = 0; i < KMAX; ++i) {
      v[i] = (i < KMAX - K) ? INFINITY : -INFINITY;
      id[i] = kNoId;
    }
  }
  __device__ __forceinline__ float thr() const { return v[KMAX - 1]; }
  // sorted insert (descending, earlier insert wins ties because columns arrive in ascending order)
  __device__ __forceinline__ void insert(float x, int xi) {
#pragma unroll
    for (int i = 0; i < KMAX; ++i) {
      const bool gt = x > v[i];
      const float tv = gt ? v[i] : x;
      const int ti = gt ? id[i] : xi;
      v[i] = gt ? x : v[i];
      id[i] = gt ? xi : id[i];
      x = tv;
      xi = ti;
    }
  }
};

// order-preserving float <-> unsigned key (0 is below every float, so a zero-filled array means "no threshold yet")
__device__ __forceinline__ uint32_t f2key(float f) {
  const uint32_t b = __float_as_uint(f);
  return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
__device__ __forceinline__ float key2f(uint32_t k) {
  return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k);
}

static constexpr int kEpiWarps = 16;   // lane quarter x 32-column part of the 128-column tile: 4 warps per SM sub-partition hide the
                                       // tcgen05.ld / shared-memory / insert-chain latencies of each other (measured: the epilogue,
                                       // not the MMA or the TMA feed, bounds this kernel)
static constexpr int kColParts = kEpiWarps / 4;
static constexpr int kAccMax = 4;    // accumulator stages in TMEM: 4 x 128 columns, or 3 when the user tile itself lives in TMEM
static constexpr int kThreads = 64 + kEpiWarps * 32;

// One 32-column chunk of one row (thread).  FAST PATH: the maxima of the four 8-column groups against the admission threshold -
// the values are never modified or copied (they stay in the registers tcgen05.ld filled).  Seen / out-of-catalog columns are
// NOT masked here: a masked column only matters if it would be admitted, and then the slow path drops it from the hit mask (a
// spurious slow-path entry costs about what masking every chunk that holds a seen item would).  SLOW PATH (a group maximum
// beats the threshold): stage that group's 8 values in shared memory so that ONE insert site serves a runtime column index,
// build the hit mask, drop masked columns, insert.
template <int KMAX>
__device__ __forceinline__ void score_chunk(const uint32_t (&raw)[32], uint32_t kill, float thr, float gthr, int col0,
                                            TopK<KMAX>& top, float* sc, bool live, uint32_t* row_thr_u) {
  // maxima of the four 8-column groups: the slow path then stages and scans only the group(s) that hold a candidate
  float g[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const float a = fmaxf(__uint_as_float(raw[8 * k]), __uint_as_float(raw[8 * k + 1]));
    const float b = fmaxf(__uint_as_float(raw[8 * k + 2]), __uint_as_float(raw[8 * k + 3]));
    const float c = fmaxf(__uint_as_float(raw[8 * k + 4]), __uint_as_float(raw[8 * k + 5]));
    const float d = fmaxf(__uint_as_float(raw[8 * k + 6]), __uint_as_float(raw[8 * k + 7]));
    g[k] = fmaxf(fmaxf(a, b), fmaxf(c, d));
  }
  const float m = fmaxf(fmaxf(g[0], g[1]), fmaxf(g[2], g[3]));
  if (m > thr) {
    const float before = top.thr();
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      if (g[k] > thr) {  // stage this group's 8 values so that ONE insert site serves a runtime column index
        uint32_t hit = 0;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          sc[i * (kEpiWarps * 32)] = __uint_as_float(raw[8 * k + i]);
          hit |= (__uint_as_float(raw[8 * k + i]) > thr) ? (1u << i) : 0u;
        }
        hit &= ~(kill >> (8 * k));
        while (hit) {
          const int i = __ffs(hit) - 1;
          hit &= hit - 1;
          const float val = sc[i * (kEpiWarps * 32)];
          if (val > fmaxf(top.thr(), gthr)) top.insert(val, col0 + 8 * k + i);
        }
      }
    }
    // publish an improved K-th best (only once the list holds K real entries, i.e. its last slot is finite)
    if (live && top.thr() > before && top.thr() > -INFINITY) atomicMax(row_thr_u, f2key(top.thr()));
  }
}


template <int KCH /* d / 64 */, int NSTAGE, int KMAX>
__global__ void __launch_bounds__(kThreads, 1)
score_topk_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                  const int32_t* __restrict__ seen_sorted, int S, int n_users, int n_items, int K, int n_splits,
                  const float* __restrict__ bias, float* __restrict__ part_vals, int32_t* __restrict__ part_ids,
                  uint32_t* __restrict__ row_thr /* [n_users] shared K-th-best keys, zero-filled */,
                  const __nv_bfloat16* __restrict__ hq_rows /* the user matrix as a plain pointer (A_TMEM) */) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sA = smem;                          // KCH chunks of 16 KB
  uint8_t* sB = smem + KCH * kChunkBytes;      // NSTAGE chunks of 16 KB
  // d = 128 / 256: the resident user tile Hq goes to TMEM (packed bf16, d/2 columns) and the MMA takes its A operand from
  // there: 73 instead of 102 cycles per 128x128x16 MMA (profiles/r1_mma_probe.md); three accumulator stages remain
  constexpr bool A_TMEM = (KCH == 2 || KCH == 4);
  constexpr int kAcc = A_TMEM ? 3 : 4;
  __shared__ uint64_t bar_a, bar_full[NSTAGE], bar_empty[NSTAGE], bar_tfull[kAccMax], bar_tempty[kAccMax];
  __shared__ uint32_t tmem_slot;
  __shared__ float s_scratch[8 * kEpiWarps * 32];  // [i][epilogue thread]: one 8-column group staged for the insert path

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int user_tile = blockIdx.x / n_splits, split = blockIdx.x % n_splits;
  const int u0 = user_tile * kTileM;
  const int n_tiles_total = (n_items + kTileN - 1) / kTileN;
  const int t_begin = (int)(((long long)n_tiles_total * split) / n_splits);
  const int t_end = (int)(((long long)n_tiles_total * (split + 1)) / n_splits);
  const int n_ct = t_end - t_begin;

  if (threadIdx.x == 0) {
    mbar_init(&bar_a, A_TMEM ? kEpiWarps : 1);
    for (int i = 0; i < NSTAGE; ++i) {
      mbar_init(&bar_full[i], 1);
      mbar_init(&bar_empty[i], 1);
    }
    for (int i = 0; i < kAcc; ++i) {
      mbar_init(&bar_tfull[i], 1);
      mbar_init(&bar_tempty[i], kEpiWarps);  // one arrive per epilogue warp
    }
    fence_barrier_init();
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
  }
  if (warp == 1) tmem_alloc(&tmem_slot, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = tmem_slot;

  if (warp == 0) {
    // ------------------------------------------------ TMA producer
    if (elect_one()) {
      if (!A_TMEM) {
        mbar_arrive_expect_tx(&bar_a, KCH * kChunkBytes);
        for (int kc = 0; kc < KCH; ++kc) tma_load_2d(sA + kc * kChunkBytes, &tmA, &bar_a, kc * 64, u0);
      }
      uint32_t it = 0;
      for (int t = t_begin; t < t_end; ++t) {
        for (int kc = 0; kc < KCH; ++kc, ++it) {
          const uint32_t s = it % NSTAGE, ph = (it / NSTAGE) & 1;
          mbar_wait(&bar_empty[s], ph ^ 1);
          mbar_arrive_expect_tx(&bar_full[s], kChunkBytes);
          tma_load_2d(sB + s * kChunkBytes, &tmB, &bar_full[s], kc * 64, t * kTileN);
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------ MMA issuer
    if (elect_one()) {
      constexpr uint32_t idesc = umma_idesc_bf16(kTileM, kTileN);
      mbar_wait(&bar_a, 0);
      tc_fence_after();
      uint32_t it = 0;
      for (int j = 0; j < n_ct; ++j) {
        const uint32_t as = j % kAcc, aph = (j / kAcc) & 1;
        mbar_wait(&bar_tempty[as], aph ^ 1);
        tc_fence_after();
        const uint32_t dcol = tmem + as * kTileN;
        for (int kc = 0; kc < KCH; ++kc, ++it) {
          const uint32_t s = it % NSTAGE, ph = (it / NSTAGE) & 1;
          mbar_wait(&bar_full[s], ph);
          tc_fence_after();
          const uint32_t a0 = smem_u32(sA + kc * kChunkBytes), b0 = smem_u32(sB + s * kChunkBytes);
#pragma unroll
          for (int ks = 0; ks < 4; ++ks) {
            if (A_TMEM)
              umma_ts(dcol, tmem + kAcc * kTileN + kc * 32 + ks * 8, umma_desc_sw128(b0 + ks * 32, 16, 1024), idesc, (kc | ks) != 0);
            else
              umma_ss(dcol, umma_desc_sw128(a0 + ks * 32, 16, 1024), umma_desc_sw128(b0 + ks * 32, 16, 1024), idesc,
                      (kc | ks) != 0);
          }
          umma_commit(&bar_empty[s]);
        }
        umma_commit(&bar_tfull[as]);
      }
    }
  } else {
    // ------------------------------------------------ epilogue: 16 warps; warp%4 = TMEM lane quarter, (warp-2)/4 = 32-column part
    const int ew = warp - 2, quarter = warp & 3, part = ew >> 2;
    const int row = quarter * 32 + lane;
    const int u = u0 + row;
    const bool live = u < n_users;
    float* sc = s_scratch + ew * 32 + lane;  // element q of this thread at sc[q * (kEpiWarps*32)]
    if (A_TMEM) {
      // thread (row, part) copies K elements [part*D/4, (part+1)*D/4) of its user row from global memory into TMEM
      constexpr int D = KCH * 64, WORDS = D / 8;   // 32-bit words (bf16 pairs) per thread
      const uint4* src = reinterpret_cast<const uint4*>(hq_rows + (size_t)(live ? u : 0) * D + part * (D / 4));
#pragma unroll
      for (int c = 0; c < WORDS; c += 16) {
        uint32_t v[16];
#pragma unroll
        for (int q = 0; q < 16; q += 4) {
          const uint4 t4 = live ? __ldg(src + ((c + q) >> 2)) : make_uint4(0u, 0u, 0u, 0u);
          v[q] = t4.x; v[q + 1] = t4.y; v[q + 2] = t4.z; v[q + 3] = t4.w;
        }
        tmem_st16(tmem + ((uint32_t)(quarter * 32) << 16) + kAcc * kTileN + part * WORDS + c, v);
      }
      tmem_st_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&bar_a);
    }
    TopK<KMAX> top;
    top.init(K);
    // cursor into this user's sorted seen list (ascending, kNoId = padding).  The next entry is prefetched one step ahead
    // so that the (rare, per thread) advance never waits on a dependent global load inside the tile loop.
    const int32_t* sp = seen_sorted ? seen_sorted + (size_t)(live ? u : 0) * S : nullptr;
    int ci = 0;
    int next_seen = kNoId, pre_seen = kNoId;
    if (sp && live) {
      const int first_col = t_begin * kTileN;
      int lo = 0, hi = S;  // lower_bound(first_col), once per CTA
      while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (sp[mid] < first_col) lo = mid + 1; else hi = mid;
      }
      ci = lo;
      next_seen = ci < S ? sp[ci] : kNoId;
      pre_seen = ci + 1 < S ? sp[ci + 1] : kNoId;
    }
    // K-th best already secured for this row by ANY thread / CTA working on it (other column halves and item splits):
    // anything strictly below it cannot reach the final top-K, so it never enters the insert path.  The shared value is
    // read one tile AHEAD (a stale threshold is only weaker, never wrong), so its L2 round trip is off the per-tile path.
    uint32_t gk = live ? *reinterpret_cast<volatile uint32_t*>(row_thr + u) : 0u;
    float gthr = -INFINITY;
    for (int t = t_begin, j = 0; t < t_end; ++t, ++j) {
      const uint32_t as = j % kAcc, aph = (j / kAcc) & 1;
      if ((j & 3) == 0) {  // refresh every 4th tile: the shared threshold moves slowly once the lists are full
        gthr = gk != 0u ? key2f(gk - 1u) : -INFINITY;  // largest value strictly below the shared K-th best
        if (live) gk = *reinterpret_cast<volatile uint32_t*>(row_thr + u);  // lands long before its use 4 tiles later
      }
      mbar_wait(&bar_tfull[as], aph);
      tc_fence_after();
      const uint32_t tbase = tmem + ((uint32_t)(quarter * 32) << 16) + as * kTileN + part * 32;
      uint32_t raw[32];
      tmem_ld32(tbase, raw);
      tmem_ld_wait();
      // the accumulator stage can be reused as soon as its values sit in registers
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&bar_tempty[as]);
      const int col0 = t * kTileN + part * 32;
      // seen items of this 32-column chunk as a bit mask (also skips entries that belong to the other column parts);
      // columns beyond the catalog (ragged last tile) are "seen" too
      uint32_t kill = 0;
      while (next_seen < col0 + 32) {
        if (next_seen >= col0) kill |= 1u << (next_seen - col0);
        next_seen = pre_seen;
        ++ci;
        pre_seen = ci + 1 < S ? sp[ci + 1] : kNoId;
      }
      if (col0 + 32 > n_items) kill |= (col0 >= n_items) ? 0xffffffffu : (0xffffffffu << (n_items - col0));
      const float thr = live ? fmaxf(top.thr(), gthr) : INFINITY;  // rows beyond the batch never enter the insert path
      if (bias == nullptr) {
        score_chunk(raw, kill, thr, gthr, col0, top, sc, live, row_thr + u);
      } else {  // biased head (BERT4Rec): warp-uniform 16-byte loads, bias padded to a multiple of 128 entries
        uint32_t xb[32];
#pragma unroll
        for (int q = 0; q < 32; q += 4) {
          const float4 b4 = __ldg(reinterpret_cast<const float4*>(bias + col0 + q));
          xb[q] = __float_as_uint(__uint_as_float(raw[q]) + b4.x);
          xb[q + 1] = __float_as_uint(__uint_as_float(raw[q + 1]) + b4.y);
          xb[q + 2] = __float_as_uint(__uint_as_float(raw[q + 2]) + b4.z);
          xb[q + 3] = __float_as_uint(__uint_as_float(raw[q + 3]) + b4.w);
        }
        score_chunk(xb, kill, thr, gthr, col0, top, sc, live, row_thr + u);
      }
    }
    if (live) {
      float* pv = part_vals + (((size_t)u * n_splits + split) * kColParts + part) * K;
      int32_t* pi = part_ids + (((size_t)u * n_splits + split) * kColParts + part) * K;
#pragma unroll
      for (int i = 0; i < KMAX; ++i)
        if (i >= KMAX - K) {
          pv[i - (KMAX - K)] = top.v[i];
          pi[i - (KMAX - K)] = top.id[i];
        }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem, 512);
}

// one warp per user: merge n_splits sorted partial lists -> final top-K; ties: smaller column first.
// Slots that no finite candidate fills (fewer than K unmasked items) are filled with the user's masked columns in
// ascending order, score -inf (torch.topk would return arbitrary -inf entries there).
__global__ void topk_merge_kernel(const float* __restrict__ part_vals, const int32_t* __restrict__ part_ids,
                                  const int32_t* __restrict__ seen_sorted, int S, int n_users, int n_items, int K,
                                  int n_splits, const int64_t* __restrict__ candidates, int64_t* __restrict__ out_ids,
                                  float* __restrict__ out_scores) {
  const int u = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (u >= n_users) return;
  const int n = n_splits * K;
  const float* pv = part_vals + (size_t)u * n;
  const int32_t* pi = part_ids + (size_t)u * n;
  // each lane owns candidates lane, lane+32, ...  ; consumed ones are flagged by setting id to kNoId+(-inf)
  float last_v = INFINITY;
  int last_id = -1;
  int n_out = 0;
  for (int k = 0; k < K; ++k) {
    // best candidate strictly after (last_v, last_id) in (score desc, id asc) order
    float bv = -INFINITY;
    int bi = kNoId;
    for (int i = lane; i < n; i += 32) {
      const float v = pv[i];
      const int id = pi[i];
      if (id == kNoId) continue;
      const bool after = (v < last_v) || (v == last_v && id > last_id);
      if (!after) continue;
      if (v > bv || (v == bv && id < bi)) {
        bv = v;
        bi = id;
      }
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
      const float ov = __shfl_xor_sync(0xffffffffu, bv, off);
      const int oi = __shfl_xor_sync(0xffffffffu, bi, off);
      if (ov > bv || (ov == bv && oi < bi)) {
        bv = ov;
        bi = oi;
      }
    }
    if (bi == kNoId) break;
    if (lane == 0) {
      out_ids[(size_t)u * K + k] = candidates ? candidates[bi] : (int64_t)bi;
      out_scores[(size_t)u * K + k] = bv;
    }
    last_v = bv;
    last_id = bi;
    ++n_out;
  }
  if (n_out < K && lane == 0) {
    int ci = 0;
    int prev = -1;
    for (int k = n_out; k < K; ++k) {
      int col = kNoId;
      while (seen_sorted && ci < S) {
        const int c = seen_sorted[(size_t)u * S + ci++];
        if (c != prev && c < n_items) {
          col = c;
          prev = c;
          break;
        }
      }
      out_ids[(size_t)u * K + k] = (col == kNoId) ? -1 : (candidates ? candidates[col] : (int64_t)col);
      out_scores[(size_t)u * K + k] = -INFINITY;
    }
  }
}

// Prepare the seen lists for score_topk: int64 ids [B,S] -> int32 columns sorted ascending, padding = kNoId.
// Ids outside [0, item_count) are padding (seen_items.py:62).  With inv_map (candidates_to_score) an id becomes its
// position in the candidate list (or padding when it is not a candidate).  One block per user, bitonic sort in smem.
template <int SPAD>
__global__ void seen_prepare_kernel(const int64_t* __restrict__ seen, int S, int item_count,
                                    const int32_t* __restrict__ inv_map, int32_t* __restrict__ out) {
  __shared__ int32_t buf[SPAD];
  const int u = blockIdx.x;
  for (int i = threadIdx.x; i < SPAD; i += blockDim.x) {
    int32_t v = kNoId;
    if (i < S) {
      const int64_t id = seen[(size_t)u * S + i];
      if (id >= 0 && id < item_count) {
        v = (int32_t)id;
        if (inv_map) {
          v = inv_map[v];
          if (v < 0) v = kNoId;
        }
      }
    }
    buf[i] = v;
  }
  __syncthreads();
  for (int k = 2; k <= SPAD; k <<= 1) {
    for (int jj = k >> 1; jj > 0; jj >>= 1) {
      for (int i = threadIdx.x; i < SPAD; i += blockDim.x) {
        const int ixj = i ^ jj;
        if (ixj > i) {
          const bool up = (i & k) == 0;
          const int32_t a = buf[i], b = buf[ixj];
          if ((a > b) == up) {
            buf[i] = b;
            buf[ixj] = a;
          }
        }
      }
      __syncthreads();
    }
  }
  for (int i = threadIdx.x; i < S; i += blockDim.x) out[(size_t)u * S + i] = buf[i];
}

static int choose_splits(int n_user_tiles, int n_item_tiles) {
  const int sms = sm_count();
  int p = sms / n_user_tiles;
  if (p < 1) p = 1;
  if (p > n_item_tiles) p = n_item_tiles;
  if (p > 64) p = 64;
  return p;
}

template <int KCH, int NSTAGE>
static int launch_score_topk(const CUtensorMap& tmA, const CUtensorMap& tmB, const int32_t* seen_sorted, int S, int B,
                             int I, int K, int n_splits, const float* bias, float* pv, int32_t* pi, uint32_t* row_thr,
                             const __nv_bfloat16* hq_rows, cudaStream_t stream) {
  const int smem = (KCH + NSTAGE) * kChunkBytes + 1024;
  const int grid = ((B + kTileM - 1) / kTileM) * n_splits;
  if (K <= 10) {
    auto kern = score_topk_kernel<KCH, NSTAGE, 10>;
    RP_CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    kern<<<grid, kThreads, smem, stream>>>(tmA, tmB, seen_sorted, S, B, I, K, n_splits, bias, pv, pi, row_thr, hq_rows);
  } else if (K <= 16) {
    auto kern = score_topk_kernel<KCH, NSTAGE, 16>;
    RP_CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    kern<<<grid, kThreads, smem, stream>>>(tmA, tmB, seen_sorted, S, B, I, K, n_splits, bias, pv, pi, row_thr, hq_rows);
  } else {
    auto kern = score_topk_kernel<KCH, NSTAGE, 32>;
    RP_CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    kern<<<grid, kThreads, smem, stream>>>(tmA, tmB, seen_sorted, S, B, I, K, n_splits, bias, pv, pi, row_thr, hq_rows);
  }
  RP_LAUNCH_CHECK();
  return RP_OK;
}

}  // namespace rp

RP_API size_t rp_score_topk_workspace(int n_users, int n_items, int d, int K) {
  (void)d;
  if (n_users <= 0 || n_items <= 0 || K <= 0) return 0;
  const int ut = (n_users + rp::kTileM - 1) / rp::kTileM, it = (n_items + rp::kTileN - 1) / rp::kTileN;
  const int p = rp::choose_splits(ut, it);
  return (size_t)n_users * p * rp::kColParts * K * 8 + (size_t)n_users * 4 + 256;
}

RP_API int rp_seen_prepare(const int64_t* seen_ids, int n_users, int S, int item_count, const int32_t* inv_map,
                    int32_t* out_sorted, void* stream_) {
  using namespace rp;
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  if (!seen_ids || !out_sorted) return RP_EINVAL;
  if (n_users <= 0 || S <= 0) return RP_ESHAPE;
  if (S <= 64) seen_prepare_kernel<64><<<n_users, 64, 0, stream>>>(seen_ids, S, item_count, inv_map, out_sorted);
  else if (S <= 256) seen_prepare_kernel<256><<<n_users, 128, 0, stream>>>(seen_ids, S, item_count, inv_map, out_sorted);
  else if (S <= 1024) seen_prepare_kernel<1024><<<n_users, 256, 0, stream>>>(seen_ids, S, item_count, inv_map, out_sorted);
  else if (S <= 4096) seen_prepare_kernel<4096><<<n_users, 512, 0, stream>>>(seen_ids, S, item_count, inv_map, out_sorted);
  else return RP_ESHAPE;
  RP_LAUNCH_CHECK();
  return RP_OK;
}

RP_API int rp_score_topk(const void* hq, const void* table, const float* bias, const int32_t* seen_sorted, int S, int n_users,
                  int n_items, int d, int K, const int64_t* candidates, int64_t* out_ids, float* out_scores,
                  void* workspace, size_t workspace_bytes, void* stream_) {
  using namespace rp;
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  if (!hq || !table || !out_ids || !out_scores || !workspace) return RP_EINVAL;
  if (n_users <= 0 || n_items <= 0 || K <= 0 || K > 32 || K > n_items) return RP_ESHAPE;
  if (d != 64 && d != 128 && d != 256 && d != 512) return RP_ESHAPE;
  if (seen_sorted && S <= 0) return RP_ESHAPE;
  if (workspace_bytes < rp_score_topk_workspace(n_users, n_items, d, K)) return RP_EWORKSPACE;
  const int ut = (n_users + kTileM - 1) / kTileM, it = (n_items + kTileN - 1) / kTileN;
  const int p = choose_splits(ut, it);
  float* pv = reinterpret_cast<float*>(workspace);
  int32_t* pi = reinterpret_cast<int32_t*>(pv + (size_t)n_users * p * kColParts * K);
  uint32_t* row_thr = reinterpret_cast<uint32_t*>(pi + (size_t)n_users * p * kColParts * K);
  RP_CUDA_CHECK(cudaMemsetAsync(row_thr, 0, (size_t)n_users * 4, stream));
  CUtensorMap tmA, tmB;
  int rc;
  if ((rc = make_tmap_bf16(&tmA, hq, n_users, d, d, 128)) != RP_OK) return rc;
  if ((rc = make_tmap_bf16(&tmB, table, n_items, d, d, 128)) != RP_OK) return rc;
  switch (d) {
    case 64: rc = launch_score_topk<1, 8>(tmA, tmB, seen_sorted, S, n_users, n_items, K, p, bias, pv, pi, row_thr,
                                            reinterpret_cast<const __nv_bfloat16*>(hq), stream); break;
    case 128: rc = launch_score_topk<2, 8>(tmA, tmB, seen_sorted, S, n_users, n_items, K, p, bias, pv, pi, row_thr,
                                            reinterpret_cast<const __nv_bfloat16*>(hq), stream); break;
    case 256: rc = launch_score_topk<4, 6>(tmA, tmB, seen_sorted, S, n_users, n_items, K, p, bias, pv, pi, row_thr,
                                            reinterpret_cast<const __nv_bfloat16*>(hq), stream); break;
    default: rc = launch_score_topk<8, 3>(tmA, tmB, seen_sorted, S, n_users, n_items, K, p, bias, pv, pi, row_thr,
                                            reinterpret_cast<const __nv_bfloat16*>(hq), stream); break;
  }
  if (rc != RP_OK) return rc;
  const int threads = 128;
  const int blocks = (n_users * 32 + threads - 1) / threads;
  topk_merge_kernel<<<blocks, threads, 0, stream>>>(pv, pi, seen_sorted, S, n_users, n_items, K, p * kColParts, candidates, out_ids,
                                                    out_scores);
  RP_LAUNCH_CHECK();
  return RP_OK;
}

