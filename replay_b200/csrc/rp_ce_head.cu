// rp_ce_head.cu - fused full-catalog cross-entropy head (training), forward and backward, without ever materialising the
// [tokens, items] logits.
//
// Replaces   logits = hidden . E^T               replay/nn/head.py:29-34, replay/nn/sequential/sasrec/model.py:258-265
//            torch.nn.CrossEntropyLoss(mean)     replay/nn/loss/ce.py:49-81 ; models/nn/sequential/sasrec/lightning.py:335-355
// and their autograd backward (dHidden, dE).
//
// Inputs are the COMPACTED valid-target rows Hc[T_v, d] (bf16, capacity T rows; T_v lives in device memory so the whole
// step stays CUDA-graph capturable), the item table E[I, d] (bf16) and labels[T_v].
//
//   ce_fwd_kernel      CTA = 128 tokens x an item split.  S = Hc.E^T tile by tile in TMEM; epilogue keeps an online
//                      (max, sum-exp) per row and picks the target logit.                      -> partial (m, s), z_y
//   ce_finalize_kernel lse, loss = mean(lse - z_y), per-token exponent offset c_t = -lse*log2e + log2(1/T_v)
//   ce_bwd_kernel<ROW> CTA = 128 tokens, loops over item tiles:   G = exp2(S*log2e + c_row) (bf16, written back into
//                      TMEM over S), dH += G . E_tile  (A from TMEM, B = the same smem tile, MN-major)
//                      final: dH[t] -= E[y_t] / T_v                                             -> dHc bf16 [T_v, d]
//   ce_bwd_kernel<COL> CTA = 128 items, loops over token tiles:   S^T = E_tile . Hc^T, G = exp2(S^T*log2e + c_col),
//                      dE += G . Hc_tile                                                          -> dE fp32 [I, d] (=)
//   ce_label_scatter   dE[y_t] -= Hc[t] / T_v   (the one-hot part of softmax - onehot, sparse)
#include <type_traits>

#include "rp_host.h"
#include "rp_gemm_desc.h"
#include "rp_sm100.cuh"

namespace rp {

static constexpr int kT = 128;                  // tile edge (rows per CTA, columns per MMA tile)
static constexpr int kChunk = 128 * 128;        // bytes of one [128 rows x 64 bf16] swizzled chunk
static constexpr float kLog2e = 1.4426950408889634f;
static constexpr float kLn2 = 0.6931471805599453f;
static constexpr int kEpiWarps = 8;
static constexpr int kThreads = 64 + kEpiWarps * 32;
// backward / fused kernels: RP_CE_BWD_CG column groups per TMEM lane quarter -> 4*CG epilogue warps (16 by default): the
// knob kept for experiments: 16 warps (CG = 4) measured ~8 % slower than 8 (CG = 2) on B200, see profiles/r1_ce_variants.md
#ifndef RP_CE_BWD_CG
#define RP_CE_BWD_CG 2
#endif
#ifndef RP_CE_ABLATE
#define RP_CE_ABLATE 0
#endif
#ifndef RP_CE_NSTAGE_D128
#define RP_CE_NSTAGE_D128 4   // B-tile ring depth of the backward / fused kernels at d = 128 (32 KB per stage)
#endif
static constexpr int kBwdCG = RP_CE_BWD_CG;
static constexpr int kBwdEpiWarps = 4 * kBwdCG;
static constexpr int kBwdThreads = 64 + kBwdEpiWarps * 32;
// RP_CE_GROUPS = 2 (d = 128): TWO such sets of epilogue warps, one per S buffer (even / odd column tiles).  One set works in
// lock step - wait, tcgen05.ld, 64 exponentials per thread, tcgen05.st, arrive - so the MUFU pipe (the 16 384 exponentials of
// a tile need >= 1024 of the ~1170 tensor cycles of the tile) idles through every load / store / barrier phase; two sets on
// different tiles fill each other's gaps (r2 ncu: MUFU 61-65 % and tensor 69-74 % busy with one set).
#ifndef RP_CE_GROUPS
#define RP_CE_GROUPS 1   /* r2 A/B (profiles/r2_ce_variants.md): two sets measured 3-5 % SLOWER than one - kept as a knob */
#endif
static constexpr int kCeMaxGroups = 2;

// tuning knobs (measured on B200, see profiles/): every RP_CE_POLY_EVERY-th exponential goes to the FMA-pipe polynomial
// instead of MUFU.EX2 (0 = MUFU only); RP_CE_NBUF3 = 1 triple-buffers S in TMEM for d <= 128.
#ifndef RP_CE_POLY_EVERY
#define RP_CE_POLY_EVERY 4   /* forward: 25 % of the exponentials on the FMA pipe (measured best, profiles/r1_ce_variants.md) */
#endif
#ifndef RP_CE_POLY_EVERY_BWD
#define RP_CE_POLY_EVERY_BWD 0   /* backward / fused passes: MUFU only (r2 A/B with the in-order issue: 0 beats 12.5 % by 2-8 %, profiles/r2_ce_variants.md) */
#endif
#ifndef RP_CE_NBUF3
#define RP_CE_NBUF3 1
#endif
#ifndef RP_CE_A_TMEM
#define RP_CE_A_TMEM 1
#endif
// MMA issue order of the backward / fused kernels (profiles/r2_ce_issue_order.md):
//   0  round-1 order: S tile j+NBUF-1 is issued right behind the second GEMM of tile j-1 and has to wait for it (its TMEM
//      buffer is the one that GEMM reads G from): the tensor pipe drains once per tile
//   1  (d <= 128) two S buffers, row tile in TMEM, S tile j+2 issued right BEHIND the second GEMM of tile j without a
//      barrier in between: tcgen05.mma instructions of one CTA execute in issue order, so the overwrite of the buffer cannot
//      overtake the reads of G; the issuing thread never waits on work it has just queued
//   2  three S buffers (row tile in shared memory), prefetch distance 1: every wait is for a GEMM issued two groups earlier
#ifndef RP_CE_ORDER
#define RP_CE_ORDER 1
#endif
#ifndef RP_CE_TN64
#define RP_CE_TN64 0      /* d <= 128: 64-wide column tiles in four S buffers (0 = 128-wide in two) */
#endif
#ifndef RP_CE_TN64_GROUPS
#define RP_CE_TN64_GROUPS 2   /* TN = 64: two epilogue warp sets on alternating tiles (1 = all 8 warps on every tile) */
#endif
#ifndef RP_CE_RELAXED_WAITS
#define RP_CE_RELAXED_WAITS 0   /* the MMA / TMA threads sleep between polls of their (long) waits: they share a sub-partition with two epilogue warps */
#endif
#ifndef RP_CE_PACE_DEPTH
#define RP_CE_PACE_DEPTH 0   /* pairs of tcgen05.mma in flight before the issuing thread waits for a completion (0 = issue at will) */
#endif
#ifndef RP_CE_NO_EMPTY
#define RP_CE_NO_EMPTY 1   /* in-order issue: stages are released by the S-complete barrier of tile j + NBUF (one commit per tile less) */
#endif
#ifndef RP_CE_PRESCALE
#define RP_CE_PRESCALE 0   /* fused pass: log2(e) folded into the TMEM row tile (one instruction less per logit; measured: no gain, 1.061 vs 1.050 ms, and the extra bf16 rounding breaks the 1e-2 gradient tolerance of test_ce_head at d = 64) */
#endif
#ifndef RP_CE_POLY_EVERY_Q1
#define RP_CE_POLY_EVERY_Q1 RP_CE_POLY_EVERY_BWD   /* polynomial share of lane quarter 1's epilogue warps (see the chunk lambda) */
#endif
#ifndef RP_CE_ISSUE_GROUP
#define RP_CE_ISSUE_GROUP 0      /* > 0: the issuing thread sleeps RP_CE_ISSUE_SLEEP_NS after every so many tcgen05.mma */
#endif
#ifndef RP_CE_ISSUE_SLEEP_NS
#define RP_CE_ISSUE_SLEEP_NS 150
#endif
#ifndef RP_CE_ISSUERS
#define RP_CE_ISSUERS 1   /* MMA-issuing threads of the backward / fused kernels (1 = warp 1 alone) */
#endif
#ifndef RP_CE_PERSIST
#define RP_CE_PERSIST 1   /* dE pass: one CTA per SM over balanced slices of the (item tile, token tile) pairs; 0 = one CTA per item tile */
#endif
#ifdef RP_CE_TRACE  // diagnostic build (-DRP_CE_TRACE): timeline of CTA 0 - 8 event kinds x the first 256 column tiles
__device__ unsigned long long g_ce_trace[2][16 * 256];   // [0]: fused forward / dH pass, [1]: dE pass; kinds 8..15: hand-over time of epilogue warp 0..7
#define RP_CTR(k, j) do { if (blockIdx.x == 0 && (j) < 256) g_ce_trace[MODE == 1][(k) * 256 + (j)] = clock64(); } while (0)
#else
#define RP_CTR(k, j) do { } while (0)
#endif
template <int DEG, int EVERY>
__device__ __forceinline__ float ce_ex2(float x, int q) {
  if (EVERY > 0 && (q % (EVERY > 0 ? EVERY : 1)) == 1) return ex2_poly<DEG>(x);
  return ex2f(x);
}

// ---- element-wise terms of the full-catalog BCE head (BCEWithLogitsLoss against a one-hot row), s = h.E_i + b_i in fp32.
// The gradient passes sum 1e4 - 1e6 sigmoids per row / column, so every term needs RELATIVE accuracy (tanh.approx-based
// sigmoids have ~2^-11 absolute error near saturation and bias those sums): e = 2^(-|s| log2 e) on MUFU.EX2, 1 / (1 + e) on
// MUFU.RCP, log1p(e) on the FMA pipe.  s = -inf (masked column / token) gives sigmoid 0 and softplus 0.
__device__ __forceinline__ float rcp_approx(float x) {
  float y;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
// log1p(e) for e in [0, 1]: e * p(e), p a degree-7 least-squares fit of log1p(e) / e (max rel. error 3.5e-7 in fp32)
__device__ __forceinline__ float log1p_unit(float e) {
  float p = fmaf(e, -0.008574675768613815f, 0.044214192777872086f);
  p = fmaf(p, e, -0.10785368084907532f);
  p = fmaf(p, e, 0.17757023870944977f);
  p = fmaf(p, e, -0.2449961155653f);
  p = fmaf(p, e, 0.3327617645263672f);
  p = fmaf(p, e, -0.49997448921203613f);
  p = fmaf(p, e, 0.9999998211860657f);
  return e * p;
}
__device__ __forceinline__ float bce_sigmoid(float s) {
  const float e = ex2f(-fabsf(s) * kLog2e);
  return (s >= 0.f ? 1.f : e) * rcp_approx(1.f + e);
}
// sigmoid(s) and softplus(s) = max(s, 0) + log1p(e^-|s|)
__device__ __forceinline__ float bce_terms(float s, float& softplus) {
  const float e = ex2f(-fabsf(s) * kLog2e);
  softplus = fmaxf(s, 0.f) + log1p_unit(e);
  return (s >= 0.f ? 1.f : e) * rcp_approx(1.f + e);
}

// ----------------------------------------------------------------------------------------------------------------
// forward
// ----------------------------------------------------------------------------------------------------------------
template <int KCH, int NSTAGE>
__global__ void __launch_bounds__(kThreads, 1)
ce_fwd_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
              const int32_t* __restrict__ n_valid_ptr, int n_items, int n_splits, const float* __restrict__ bias,
              float2* __restrict__ part /* [T, n_splits, 2] (m in log2 units, s) */,
              const int32_t* __restrict__ skip_if_safe) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sA = smem;
  uint8_t* sB = smem + KCH * kChunk;
  __shared__ uint64_t bar_a, bar_full[NSTAGE], bar_empty[NSTAGE], bar_tfull[2], bar_tempty[2];
  __shared__ uint32_t tmem_slot;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int tok_tile = blockIdx.x / n_splits, split = blockIdx.x % n_splits;
  if (skip_if_safe && *skip_if_safe != 0) return;  // the fused pass covers this step
  const int n_valid = *n_valid_ptr;
  const int t0 = tok_tile * kT;
  if (t0 >= n_valid) return;  // uniform for the CTA
  const int n_tiles_total = (n_items + kT - 1) / kT;
  const int j_begin = (int)(((long long)n_tiles_total * split) / n_splits);
  const int j_end = (int)(((long long)n_tiles_total * (split + 1)) / n_splits);

  if (threadIdx.x == 0) {
    mbar_init(&bar_a, 1);
    for (int i = 0; i < NSTAGE; ++i) {
      mbar_init(&bar_full[i], 1);
      mbar_init(&bar_empty[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&bar_tfull[i], 1);
      mbar_init(&bar_tempty[i], kEpiWarps);
    }
    fence_barrier_init();
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
  }
  if (warp == 1) tmem_alloc(&tmem_slot, 256);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = tmem_slot;

  if (warp == 0) {
    if (elect_one()) {
      mbar_arrive_expect_tx(&bar_a, KCH * kChunk);
      for (int kc = 0; kc < KCH; ++kc) tma_load_2d(sA + kc * kChunk, &tmA, &bar_a, kc * 64, t0);
      uint32_t it = 0;
      for (int j = j_begin; j < j_end; ++j)
        for (int kc = 0; kc < KCH; ++kc, ++it) {
          const uint32_t s = it % NSTAGE, ph = (it / NSTAGE) & 1;
          mbar_wait(&bar_empty[s], ph ^ 1);
          mbar_arrive_expect_tx(&bar_full[s], kChunk);
          tma_load_2d(sB + s * kChunk, &tmB, &bar_full[s], kc * 64, j * kT);
        }
    }
  } else if (warp == 1) {
    if (elect_one()) {
      constexpr uint32_t idesc = umma_idesc_bf16(kT, kT);
      mbar_wait(&bar_a, 0);
      tc_fence_after();
      uint32_t it = 0;
      for (int j = j_begin, n = 0; j < j_end; ++j, ++n) {
        const uint32_t as = n & 1, aph = (n >> 1) & 1;
        mbar_wait(&bar_tempty[as], aph ^ 1);
        tc_fence_after();
        const uint32_t dcol = tmem + as * kT;
        for (int kc = 0; kc < KCH; ++kc, ++it) {
          const uint32_t s = it % NSTAGE, ph = (it / NSTAGE) & 1;
          mbar_wait(&bar_full[s], ph);
          tc_fence_after();
          const uint32_t a0 = smem_u32(sA + kc * kChunk), b0 = smem_u32(sB + s * kChunk);
#pragma unroll
          for (int ks = 0; ks < 4; ++ks)
            umma_ss(dcol, umma_desc_sw128(a0 + ks * 32, 16, 1024), umma_desc_sw128(b0 + ks * 32, 16, 1024), idesc,
                    (kc | ks) != 0);
          umma_commit(&bar_empty[s]);
        }
        umma_commit(&bar_tfull[as]);
      }
    }
  } else {
    const int ew = warp - 2, quarter = warp & 3, half = ew >> 2;
    const int row = quarter * 32 + lane;
    const int t = t0 + row;
    float m = -1e30f, ssum = 0.f;  // m in log2 units
    for (int j = j_begin, n = 0; j < j_end; ++j, ++n) {
      const uint32_t as = n & 1, aph = (n >> 1) & 1;
      mbar_wait(&bar_tfull[as], aph);
      tc_fence_after();
      const uint32_t tbase = tmem + ((uint32_t)(quarter * 32) << 16) + as * kT + half * 64;
      uint32_t raw[64];
      tmem_ld32(tbase, *reinterpret_cast<uint32_t(*)[32]>(&raw[0]));
      tmem_ld32(tbase + 32, *reinterpret_cast<uint32_t(*)[32]>(&raw[32]));
      tmem_ld_wait();
      // the accumulator stage is free as soon as its values sit in registers
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&bar_tempty[as]);
      const int col0 = j * kT + half * 64;
      if (bias) {  // untied / biased head (BERT4Rec): logits = h.W^T + b ; warp-uniform 16-byte loads (bias is padded to 128)
#pragma unroll
        for (int q = 0; q < 64; q += 4) {
          const float4 b4 = __ldg(reinterpret_cast<const float4*>(bias + col0 + q));
          raw[q + 0] = __float_as_uint(__uint_as_float(raw[q + 0]) + b4.x);
          raw[q + 1] = __float_as_uint(__uint_as_float(raw[q + 1]) + b4.y);
          raw[q + 2] = __float_as_uint(__uint_as_float(raw[q + 2]) + b4.z);
          raw[q + 3] = __float_as_uint(__uint_as_float(raw[q + 3]) + b4.w);
        }
      }
      if (col0 + 64 > n_items) {  // ragged last tile
#pragma unroll
        for (int q = 0; q < 64; ++q)
          if (col0 + q >= n_items) raw[q] = 0xff800000u;  // -inf
      }
      float cm0 = __uint_as_float(raw[0]), cm1 = __uint_as_float(raw[1]);
#pragma unroll
      for (int q = 2; q < 64; q += 2) {
        cm0 = fmaxf(cm0, __uint_as_float(raw[q]));
        cm1 = fmaxf(cm1, __uint_as_float(raw[q + 1]));
      }
      const float mn = fmaxf(m, fmaxf(cm0, cm1) * kLog2e);
      ssum *= ex2f(m - mn);
      m = mn;
      // half of the exponentials on MUFU, half on the FMA pipe
      float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
#pragma unroll
      for (int q = 0; q < 64; q += 4) {
        a0 += ce_ex2<4, RP_CE_POLY_EVERY>(fmaf(__uint_as_float(raw[q + 0]), kLog2e, -mn), q + 0);
        a1 += ce_ex2<4, RP_CE_POLY_EVERY>(fmaf(__uint_as_float(raw[q + 1]), kLog2e, -mn), q + 1);
        a2 += ce_ex2<4, RP_CE_POLY_EVERY>(fmaf(__uint_as_float(raw[q + 2]), kLog2e, -mn), q + 2);
        a3 += ce_ex2<4, RP_CE_POLY_EVERY>(fmaf(__uint_as_float(raw[q + 3]), kLog2e, -mn), q + 3);
      }
      ssum += (a0 + a1) + (a2 + a3);
    }
    if (t < n_valid) part[((size_t)t * n_splits + split) * 2 + half] = make_float2(m, ssum);
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem, 256);
}

// Per-row variants of the full-catalog head (all single positive label per position):
//   w_ext   sample weights of the valid targets (compacted order): loss = mean_t w_t ce_t
//           replay/nn/loss/logout_ce.py:148-228 LogOutCEWeighted ; replay/nn/loss/ce.py:84-143 CEWeighted
//   kind 1  LogInCE (replay/nn/loss/login_ce.py:170-239): loss_t = -clamp(log(p_t + eps), -c, c), p_t = softmax prob of
//           the positive; its gradient is the CE gradient of the row times p / (p + eps) (0 where the clamp is active)
// Both act as a per-row factor w_t on (softmax - onehot) / T_v: the forward's finalisation writes it to roww[t], folds it into
// the exponent offset cvec[t] = -lse2 + log2(w_t / T_v) the gradient passes exponentiate with, and the one-hot terms read it.
struct CeRowOpts {
  const float* w_ext;    // [capacity] or null
  float* roww;           // [capacity] gradient weight per row (workspace); null only for the plain head without workspace
  int kind;              // 0 CE, 1 LogInCE
  float log_eps, clamp;
};
// row loss and gradient weight from the log-sum-exp (natural log) and the target logit
__device__ __forceinline__ void ce_row_terms(const CeRowOpts& o, int t, float lse, float zy, float& row_loss, float& wg) {
  const float wx = o.w_ext ? o.w_ext[t] : 1.f;
  float lt = lse - zy;
  wg = wx;
  if (o.kind == 1) {
    const float pr = __expf(zy - lse);
    const float lg = __logf(pr + o.log_eps);
    lt = -fminf(fmaxf(lg, -o.clamp), o.clamp);
    wg *= (lg > -o.clamp && lg < o.clamp) ? pr / (pr + o.log_eps) : 0.f;
  }
  row_loss = wx * lt;
}

// lse / loss / per-token exponent offsets.  One warp per token: merges the (max, sum) partials, computes the target logit
// z_y = hc[t] . E[y_t] as a gather-dot (keeps the per-element target pick out of the MMA epilogue), accumulates the loss.
// Deterministic: per-block partial sums, the last block adds them in index order.
__global__ void ce_finalize_kernel(const float2* __restrict__ part, const __nv_bfloat16* __restrict__ hc,
                                   const __nv_bfloat16* __restrict__ table, const int32_t* __restrict__ labels,
                                   const float* __restrict__ bias, const int32_t* __restrict__ n_valid_ptr, int n_part,
                                   int capacity, int d,
                                   float* __restrict__ lse_out, float* __restrict__ cvec, float* __restrict__ block_sums,
                                   unsigned int* __restrict__ ticket, float* __restrict__ loss_out,
                                   const int32_t* __restrict__ skip_if_safe, const CeRowOpts row) {
  if (skip_if_safe && *skip_if_safe != 0) return;
  const int n_valid = *n_valid_ptr;
  const float inv_n = n_valid > 0 ? 1.f / (float)n_valid : 0.f;
  const int lane = threadIdx.x & 31, wpb = blockDim.x >> 5;
  float local = 0.f;
  for (int t = blockIdx.x * wpb + (threadIdx.x >> 5); t < capacity; t += gridDim.x * wpb) {
    if (t < n_valid) {
      const float2* p = part + (size_t)t * n_part;
      float M = -1e30f;
      for (int i = lane; i < n_part; i += 32) M = fmaxf(M, p[i].x);
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) M = fmaxf(M, __shfl_xor_sync(0xffffffffu, M, o));
      float S = 0.f;
      for (int i = lane; i < n_part; i += 32) S += p[i].y * exp2f(p[i].x - M);
      const __nv_bfloat16* hr = hc + (size_t)t * d;
      const __nv_bfloat16* er = table + (size_t)labels[t] * d;
      float z = 0.f;
      for (int c = lane * 2; c < d; c += 64) {
        const float2 a = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(hr + c));
        const float2 b = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(er + c));
        z = fmaf(a.x, b.x, z);
        z = fmaf(a.y, b.y, z);
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        S += __shfl_xor_sync(0xffffffffu, S, o);
        z += __shfl_xor_sync(0xffffffffu, z, o);
      }
      if (bias) z += bias[labels[t]];
      const float lse2 = M + log2f(S);  // log2 units
      const float lse = lse2 * kLn2;
      if (lane == 0) {
        float rl, wg;
        ce_row_terms(row, t, lse, z, rl, wg);
        lse_out[t] = lse;
        cvec[t] = -lse2 + log2f(wg * inv_n);
        if (row.roww) row.roww[t] = wg;
        local += rl;
      }
    } else if (lane == 0) {
      cvec[t] = -INFINITY;  // rows beyond T_v contribute nothing to the backward
    }
  }
  __shared__ float red[32];
  __shared__ bool last;
  if (lane == 0) red[threadIdx.x >> 5] = local;
  __syncthreads();
  if (threadIdx.x == 0) {
    float s = 0.f;
    for (int i = 0; i < wpb; ++i) s += red[i];
    block_sums[blockIdx.x] = s;
    __threadfence();
    last = (atomicAdd(ticket, 1u) == gridDim.x - 1);
  }
  __syncthreads();
  if (last && threadIdx.x == 0) {
    __threadfence();
    float s = 0.f;
    for (int i = 0; i < (int)gridDim.x; ++i) s += reinterpret_cast<volatile float*>(block_sums)[i];
    loss_out[0] = s * inv_n;  // mean over valid targets
    loss_out[1] = inv_n;
  }
}

// Direct completion of the fused pass when the catalog is NOT split over CTAs (n_splits == 1: the CTA has seen every item of
// its 128 tokens): lse, exponent offsets, per-row loss terms and the final bf16 dH are written from the accumulator itself, so
// the partial-gradient round trip through HBM (2 x T_v x d fp32) and ce_fused_finalize_kernel disappear.
struct CeDirect {
  __nv_bfloat16* d_hc;   // null: column-split mode (partials + ce_fused_finalize_kernel)
  float* lse;
  float* cvec;
  float* row_loss;       // [capacity] weighted row losses; summed in a fixed order by ce_loss_reduce_kernel
  CeRowOpts row;         // (row.roww is also what MODE 0 scales its one-hot term with)
  int use_lse_off;       // fused pass as the FALLBACK's gradient pass: exponent offset of row t = -lse[t] (from the two-pass
                         // forward) instead of the fixed reference 0, so G is the softmax itself (z ~ 1) whatever |logit| is
};

// loss = mean over the valid targets of row_loss, deterministic (fixed partition + tree); also publishes 1 / T_v
__global__ void __launch_bounds__(1024) ce_loss_reduce_kernel(const float* __restrict__ row_loss, const int32_t* __restrict__ n_valid_ptr,
                                                              const int32_t* __restrict__ safe_flag, float* __restrict__ loss_out,
                                                              int run_if_safe) {
  if (safe_flag && (*safe_flag != 0) != (run_if_safe != 0)) return;
  __shared__ float red[1024];
  const int n_valid = *n_valid_ptr;
  float a = 0.f;
  for (int i = threadIdx.x; i < n_valid; i += 1024) a += row_loss[i];
  red[threadIdx.x] = a;
  __syncthreads();
  for (int o = 512; o > 0; o >>= 1) {
    if ((int)threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    const float inv_n = n_valid > 0 ? 1.f / (float)n_valid : 0.f;
    loss_out[0] = red[0] * inv_n;
    loss_out[1] = inv_n;
  }
}

// ----------------------------------------------------------------------------------------------------------------
// backward (both directions share one kernel)
//   COLCONST = false : rows = tokens (A = Hc tile), columns = items  -> acc = dHc tile [128, d]
//   COLCONST = true  : rows = items  (A = E tile),  columns = tokens -> acc = dE tile  [128, d]
// ----------------------------------------------------------------------------------------------------------------
// MODE 0: rows = tokens, G = softmax/T_v from the stored lse (two-pass fallback)      -> out = dHc bf16
// MODE 1: rows = items (COLCONST), columns = tokens                                    -> out = dE fp32
// MODE 2: rows = tokens, FUSED forward+backward: G~ = exp(s + b) with reference max 0 (valid while |s| is bounded, see
//         ce_bound_kernel), per-row sum of G~ and un-normalised dH~ = sum_i G~ E_i over this CTA's column split
//                                                                                      -> out = partial dH~ fp32, zpart
// One SEGMENT of a CTA's work = one row tile against a contiguous run of column tiles.  The per-row-tile launches (fused
// forward / two-pass dH: grid = row tiles x column splits) have exactly one segment per CTA.  The dE pass is PERSISTENT: the
// grid is one CTA per SM and CTA c owns the slice [W c / G, W (c+1) / G) of the W = row tiles x column tiles linearised
// (row tile, column tile) pairs - up to a few segments, every SM busy to the last tile (391 item tiles as one CTA each were
// 2.64 waves on 148 SMs: 12 % of the pass was an idle tail).  A segment that does not cover its row tile's whole column
// range adds its partial accumulator to the (zeroed) output with vector reductions.
struct CeSeg {
  long long w, w_end;
  int n_ct_all, row_tile, j0, n;
  bool valid;
  __device__ void set() {
    valid = w < w_end;
    row_tile = (int)(w / n_ct_all);
    j0 = (int)(w - (long long)row_tile * n_ct_all);
    const long long left = w_end - w;
    n = (n_ct_all - j0 < left) ? n_ct_all - j0 : (int)left;
  }
  __device__ void advance() {
    w += n;
    set();
  }
};

// TN = width of a column tile (= of one S buffer in TMEM).  TN = 64 with FOUR S buffers (d <= 128): the chain
//   first GEMM (S) -> epilogue (G over S) -> second GEMM (reads G) -> first GEMM of the tile that reuses the buffer
// is serial per buffer, so with two 128-wide buffers a tile took (tensor time + epilogue time + hand-off latencies) / 2 =
// ~1535 cycles although the tensor pipe and the MUFU pipe were each busy for only 1024 of them (ncu r2i: both 67 %).  Four
// 64-wide buffers use the same 256 TMEM columns, keep four such chains in flight, and leave S of the next tile complete long
// before the epilogue gets to it (so its first TMEM load can be issued ahead of time).
// CG / GROUPS = how the 8 epilogue warps divide the work.  TN = 128: CG = 2 column groups per TMEM lane quarter, all 8 warps
// on every tile.  TN = 64: TWO warp SETS (GROUPS = 2) of one warp per lane quarter (CG = 1), set g owns the tiles j = g mod 2.
// The timeline of a CTA (tools/trace_ce.py, profiles/r2_ce_timeline.md) shows ~450 cycles per tile in the epilogue that are
// not exponentials - waking up on the S barrier, the first TMEM load, the drain of the last exponentials into the TMEM store,
// the hand-over - next to 16 cycles per column of MUFU time (two warps share a sub-partition's MUFU).  With one set these
// phases are serial (1500 cycles per 128 columns, MUFU 67 % busy); with two sets on different tiles the sub-partition's two
// warps are out of phase and the other warp's exponentials fill them.
// NI = number of MMA-issuing threads (warp 1 and the warps behind the epilogue warps, one per SM sub-partition).  Issuing a
// tile's 16 tcgen05.mma keeps the issuing thread's sub-partition from issuing anything else for ~700 cycles (timeline: the
// two epilogue warps that share warp 1's sub-partition handed their G over 700-900 cycles after the other six, and the tile
// pace followed them).  NI = 3 issuers take the tiles round-robin, so sub-partitions 1-3 lose a third of that each (sub-
// partition 0 hosts the TMA thread); an mbarrier token passes the right to issue from tile to tile, which keeps the
// instructions in tile order in the (in-order) tensor pipe.
// BCE = true: the loss policy of the full-catalog BCE head (rp_bce_head_*) on the same pipeline, with other epilogues -
//   MODE 2: G = sigmoid(s + b_i) instead of the exponential, row sums of softplus(s + b_i) instead of those of G; columns
//           >= n_items are masked explicitly (a zero-filled item row is s = b_i, not -inf); the direct finish writes
//           dH = acc / T_v - E[y] / T_v and the row loss sum_i softplus - s_y (no normaliser, no lse, no bound)
//   MODE 1: G = sigmoid(s + b_row + cvec[col]) with cvec = 0 for the valid tokens and -inf beyond (the bias cannot be pulled
//           out as a row factor e^{b_i} as it is for CE); dE = acc / T_v, d_bias = sum of G / T_v
template <int KCH, int NSTAGE, int MODE, int NBUF, bool A_TMEM, bool INORDER, bool HAS_BIAS, int GROUPS, bool PERSIST, int TN, int CG, int NI,
          bool BCE>
__global__ void __launch_bounds__(64 + GROUPS * 4 * CG * 32 + (NI - 1) * 32, 1)
ce_bwd_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
              const __nv_bfloat16* __restrict__ a_rows /* the row-side matrix (tmA) as a plain pointer, for A_TMEM */,
              const float* __restrict__ cvec /* [T] exponent offsets per token */, const int32_t* __restrict__ labels,
              const __nv_bfloat16* __restrict__ table, const float* __restrict__ loss_inv /* [1] = 1/T_v */,
              const int32_t* __restrict__ n_valid_ptr, int n_items, const float* __restrict__ bias,
              float* __restrict__ d_bias, void* __restrict__ out, const int32_t* __restrict__ safe_flag, int run_if_safe,
              int n_splits, int capacity, float* __restrict__ zpart, const CeDirect direct) {
  constexpr bool COLCONST = (MODE == 1);
  constexpr bool FUSED = (MODE == 2);
  constexpr int kW = TN / CG;  // S columns owned by one epilogue warp (its bf16 G lands in the first kW/2 of them)
  constexpr int kChunkB = TN * 128;   // bytes of one [TN rows x 64 bf16] swizzled chunk of a column tile
  // fused pass with the row tile in TMEM and no bias: the tile is multiplied by log2(e) on its way into TMEM, so a logit's
  // exponential is ONE instruction (ex2 of the accumulator word: live rows have offset 0) instead of FFMA + ex2 - the
  // epilogue warps next to the MMA-issuing thread are short of issue slots (profiles/r2_ce_timeline.md)
  constexpr bool PRESCALE = FUSED && A_TMEM && !HAS_BIAS && !BCE && (RP_CE_PRESCALE != 0);
  constexpr int kEW = 4 * CG * GROUPS;   // epilogue warps in total
  constexpr int kSlots = CG * GROUPS;      // column slots of the accumulator read-out / of the row-sum partials
  static_assert(GROUPS == 1 || (GROUPS == 2 && NBUF % 2 == 0), "two epilogue warp sets: even / odd S buffers");
  static_assert(NBUF * TN + KCH * 64 + (A_TMEM ? KCH * 32 : 0) <= 512, "TMEM: S buffers + accumulator + row tile");
  constexpr int D = KCH * 64;
  if (safe_flag && (*safe_flag != 0) != (run_if_safe != 0)) return;  // fused path vs two-pass fallback (uniform)
  constexpr int kStage = KCH * kChunkB;   // one column tile in shared memory
  constexpr int kATile = KCH * kChunk;    // the row tile (when it is not in TMEM)
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  // A_TMEM: the resident row tile lives in TMEM (K-major, two bf16 per 32-bit column) and the first GEMM reads it from
  // there, which halves that GEMM's shared-memory traffic - M=128 x N=128 SS MMAs need the full 128 B/clk of smem.
  uint8_t* sA = smem;
  uint8_t* sB = smem + (A_TMEM ? 0 : kATile);
  __shared__ __align__(16) float s_cc[NSTAGE][TN];
  __shared__ float s_gsum[kSlots][kT];
  __shared__ float s_dot[FUSED ? kSlots : 1][kT];
  // S-complete barriers form a ring over the smem STAGES (not the NBUF TMEM buffers): the TMA thread, which runs up to
  // NSTAGE tiles ahead, can then wait for one particular tile's first GEMM without its phase being lapped (see NO_EMPTY)
  __shared__ uint64_t bar_a, bar_full[NSTAGE], bar_empty[NSTAGE], bar_sfull[NSTAGE], bar_sfree[NBUF], bar_pfull[NBUF], bar_acc, bar_tok[NI], bar_pace[8];
  // NO_EMPTY: with the in-order issue a tile's smem stage is free once the first GEMM of tile j + NBUF has completed (it is
  // queued right behind the second GEMM of tile j, the stage's last reader) - the S-complete barrier of that tile doubles as
  // the stage-free signal and the tcgen05.commit on bar_empty (~50 cycles per tile, profiles/r2_ce_timeline.md) goes away
  constexpr bool NO_EMPTY = INORDER && NI == 1 && (NSTAGE > NBUF + 1) && (RP_CE_NO_EMPTY != 0);
  __shared__ uint32_t tmem_slot;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n_valid = *n_valid_ptr;
  static_assert(!PERSIST || (COLCONST && A_TMEM), "persistent work slices: dE pass with the row tile in TMEM");
  const int split = FUSED ? blockIdx.x % n_splits : 0;
  const int n_rows = COLCONST ? n_items : n_valid;
  const int n_cols = COLCONST ? n_valid : n_items;
  const int n_ct_all = (n_cols + TN - 1) / TN;              // column tiles of the whole problem
  const int jg0 = FUSED ? (int)(((long long)n_ct_all * split) / n_splits) : 0;        // first column tile of this CTA
  CeSeg seg0;
  seg0.n_ct_all = n_ct_all > 0 ? n_ct_all : 1;
  if (PERSIST) {
    const long long W = (long long)((n_rows + kT - 1) / kT) * n_ct_all;
    seg0.w = W * blockIdx.x / gridDim.x;
    seg0.w_end = W * (blockIdx.x + 1) / gridDim.x;
    seg0.set();
    if (!seg0.valid) return;   // (uniform) nothing to do: the output was zeroed by the host side
  } else {
    seg0.row_tile = FUSED ? blockIdx.x / n_splits : blockIdx.x;
    seg0.j0 = jg0;
    seg0.n = FUSED ? (int)(((long long)n_ct_all * (split + 1)) / n_splits) - jg0 : n_ct_all;
    seg0.w = 0;
    seg0.w_end = seg0.n;       // advance() ends the iteration after this one segment (n = 0 included)
    seg0.valid = true;
    if (seg0.row_tile * kT >= n_rows) return;
  }

  if (threadIdx.x == 0) {
    mbar_init(&bar_a, A_TMEM ? kEW : 1);
    for (int i = 0; i < NSTAGE; ++i) {
      mbar_init(&bar_full[i], 1);
      mbar_init(&bar_empty[i], 1);
    }
    for (int i = 0; i < NSTAGE; ++i) mbar_init(&bar_sfull[i], 1);
    for (int i = 0; i < NBUF; ++i) {
      mbar_init(&bar_sfree[i], 1);
      mbar_init(&bar_pfull[i], 4 * CG);
    }
    mbar_init(&bar_acc, 1);
    for (int i = 0; i < NI; ++i) mbar_init(&bar_tok[i], 1);
    for (int i = 0; i < 8; ++i) mbar_init(&bar_pace[i], 1);
    fence_barrier_init();
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
  }
  if (warp == 1) tmem_alloc(&tmem_slot, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = tmem_slot;
  const uint32_t tmem_acc = tmem + NBUF * TN;   // S buffers first, then the [128 x D] accumulator
  const uint32_t tmem_a = tmem_acc + D;         // A_TMEM: [128 x D] bf16 operand, D/2 columns

  if (warp == 0) {
    if (elect_one()) {
      if (!A_TMEM) {
        mbar_arrive_expect_tx(&bar_a, kATile);
        for (int kc = 0; kc < KCH; ++kc) tma_load_2d(sA + kc * kChunk, &tmA, &bar_a, kc * 64, seg0.row_tile * kT);
      }
      // the column-tile ring runs on a tile counter that continues across segments: the loads of the next segment's first
      // tiles are already in flight while the current segment drains
      uint32_t g = 0;
      for (CeSeg sg = seg0; sg.valid; sg.advance())
        for (int jl = 0; jl < sg.n; ++jl, ++g) {
          const uint32_t s = g % NSTAGE, ph = (g / NSTAGE) & 1;
          const int jc = sg.j0 + jl;   // column tile
          if (NO_EMPTY) {
            // stage s was last used by tile g - NSTAGE; it is free when S of tile g - NSTAGE + NBUF is complete
            if (g >= (uint32_t)NSTAGE) {
              const uint32_t w = g - NSTAGE + NBUF;
              mbar_wait(&bar_sfull[w % NSTAGE], (w / NSTAGE) & 1);
            }
          } else {
#if RP_CE_RELAXED_WAITS
            mbar_wait_relaxed(&bar_empty[s], ph ^ 1);
#else
            mbar_wait(&bar_empty[s], ph ^ 1);
#endif
          }
          mbar_arrive_expect_tx(&bar_full[s], kStage + (COLCONST ? TN * 4 : 0));
          for (int kc = 0; kc < KCH; ++kc)
            tma_load_2d(sB + s * kStage + kc * kChunkB, &tmB, &bar_full[s], kc * 64, jc * TN);
          if (COLCONST) {
            asm volatile(
                "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                    smem_u32(&s_cc[s][0])),
                "l"(cvec + (size_t)jc * TN), "r"(TN * 4), "r"(smem_u32(&bar_full[s]))
                : "memory");
          }
        }
    }
  } else if (warp == 1 || warp >= 2 + kEW) {
    const int ii = warp == 1 ? 0 : warp - (2 + kEW) + 1;   // issuer index: tiles with (ring position) % NI == ii are mine
    if (elect_one()) {
      constexpr uint32_t idesc1 = umma_idesc_bf16(kT, TN);
      constexpr uint32_t idesc2 = umma_idesc_bf16(kT, D, false, true);
      // PRE S tiles are in flight ahead of the second GEMM.  INORDER: tile j+NBUF follows the second GEMM of tile j through
      // the in-order tensor pipe (no barrier); otherwise tile j+PRE is issued before it and waits for the second GEMM of
      // tile j+PRE-NBUF (RP_CE_ORDER 0: the one issued last -> pipe drain; 2: two groups back)
      constexpr int PRE = INORDER ? NBUF : ((RP_CE_ORDER == 2 && NBUF >= 3) ? NBUF - 2 : NBUF - 1);
      uint32_t g0 = 0, nseg = 0;   // ring position of the segment's first tile (S buffers, smem stages); segment count
      uint32_t n_tok = 0;          // tokens this issuer has consumed (parity of its token barrier)
      // Issue pacing.  The tensor pipe's instruction queue holds ~6 tcgen05.mma; a further one does not just make this thread
      // wait - it stalls the DISPATCH of this thread's SM sub-partition, and the two epilogue warps that live there with it
      // (timeline, tools/trace_ce.py: their hand-over came 700-900 cycles after the other six warps', whichever sub-partition
      // the issuer was moved to).  So instructions go out in pairs, each pair committed to a ring of eight mbarriers, and pair
      // m is only issued once pair m - DEPTH has completed: the waiting happens on an mbarrier (harmless) instead of in the
      // dispatch stage, and the pipe still has 2 (DEPTH - 1) .. 2 DEPTH instructions queued.
      constexpr uint32_t DEPTH = RP_CE_PACE_DEPTH;
      uint32_t n_pair = 0, n_half = 0;
      // Open-loop variant (RP_CE_ISSUE_GROUP / RP_CE_ISSUE_SLEEP_NS): after every GROUP instructions the issuing thread
      // sleeps (nanosleep deschedules the warp: the sub-partition's dispatch is free) for about the time the pipe needs to
      // drain them, instead of sitting in the dispatch stage until the queue has room.
      uint32_t n_issued = 0;
      auto pace = [&]() {          // call right before every tcgen05.mma
        if (RP_CE_ISSUE_GROUP > 0 && NI == 1) {
          if (n_issued != 0 && n_issued % RP_CE_ISSUE_GROUP == 0) __nanosleep(RP_CE_ISSUE_SLEEP_NS);
          ++n_issued;
        }
        if (DEPTH == 0 || NI > 1) return;
        if ((n_half & 1) == 0 && n_pair >= DEPTH) {
          const uint32_t m = n_pair - DEPTH;
          mbar_wait(&bar_pace[m & 7], (m >> 3) & 1);
        }
      };
      auto paced = [&]() {         // call right after every tcgen05.mma
        if (DEPTH == 0 || NI > 1) return;
        if (n_half & 1) {
          umma_commit(&bar_pace[n_pair & 7]);
          ++n_pair;
        }
        ++n_half;
      };
      for (CeSeg sg = seg0; sg.valid; sg.advance(), ++nseg) {
        const int n_ct = sg.n;
        auto issue_mma1 = [&](int jl) {
          const uint32_t g = g0 + jl, s = g % NSTAGE, ph = (g / NSTAGE) & 1;
          mbar_wait(&bar_full[s], ph);
          if (!INORDER && g >= NBUF) mbar_wait(&bar_sfree[g % NBUF], ((g / NBUF) - 1) & 1);
          tc_fence_after();
          const uint32_t dcol = tmem + (g % NBUF) * TN;
#pragma unroll
          for (int kc = 0; kc < KCH; ++kc) {
            const uint32_t a0 = smem_u32(sA + kc * kChunk), b0 = smem_u32(sB + s * kStage + kc * kChunkB);
#pragma unroll
            for (int ks = 0; ks < 4; ++ks) {
              pace();
              if (A_TMEM)
                umma_ts(dcol, tmem_a + kc * 32 + ks * 8, umma_desc_sw128(b0 + ks * 32, 16, 1024), idesc1, (kc | ks) != 0);
              else
                umma_ss(dcol, umma_desc_sw128(a0 + ks * 32, 16, 1024), umma_desc_sw128(b0 + ks * 32, 16, 1024), idesc1,
                        (kc | ks) != 0);
              paced();
            }
          }
          umma_commit(&bar_sfull[g % NSTAGE]);
        };
        for (int jl = 0; jl < n_ct; ++jl) {
          const uint32_t g = g0 + jl, s = g % NSTAGE;
          if (NI > 1) {
            if ((int)(g % NI) != ii) continue;
            if (g > 0) {   // the right to issue: the issuer of tile g-1 has queued all of its instructions
              mbar_wait(&bar_tok[ii], n_tok & 1);
              ++n_tok;
              tc_fence_after();
            }
          }
          if (jl == 0) {
            // the row tile of this segment is in place (TMEM: written by the epilogue warps after they drained the previous
            // segment's accumulator, so the accumulator may be overwritten as well); the segment's first S tiles go first
            mbar_wait(&bar_a, nseg & 1);
            tc_fence_after();
            for (int q = 0; q < PRE && q < n_ct; ++q) issue_mma1(q);
          }
          if (!INORDER && jl + PRE < n_ct) issue_mma1(jl + PRE);
          RP_CTR(4, g);   // MMA thread starts waiting for G of tile g
#if RP_CE_RELAXED_WAITS
          mbar_wait_relaxed(&bar_pfull[g % NBUF], (g / NBUF) & 1);
#else
          mbar_wait(&bar_pfull[g % NBUF], (g / NBUF) & 1);
#endif
          RP_CTR(5, g);   // ... G of tile g is there
          tc_fence_after();
          const uint32_t pcol = tmem + (g % NBUF) * TN;  // G (bf16 pairs) lives over S, kW/2 packed columns per column group
          const uint32_t b0 = smem_u32(sB + s * kStage);
#pragma unroll
          for (int ks = 0; ks < TN / 16; ++ks) {
            pace();
            umma_ts(tmem_acc, pcol + ((ks * 16) / kW) * kW + ((ks * 16) % kW) / 2, umma_desc_sw128(b0 + ks * 2048, kChunkB, 1024),
                    idesc2, (jl | ks) != 0);
            paced();
          }
          if (!NO_EMPTY) umma_commit(&bar_empty[s]);
          if (INORDER) {
            if (jl + PRE < n_ct) issue_mma1(jl + PRE);
          } else {
            umma_commit(&bar_sfree[g % NBUF]);
          }
          if (jl == n_ct - 1) umma_commit(&bar_acc);   // (in-order pipe: everything issued before it has completed as well)
          RP_CTR(6, g);   // second GEMM of tile g and first GEMM of tile g + PRE are queued
          if (NI > 1) {
            tc_fence_before();
            mbar_arrive(&bar_tok[(g + 1) % NI]);
          }
        }
        if (n_ct == 0 && ii == 0) {   // (single-segment launches only) nothing to multiply: release the epilogue's final wait
          mbar_wait(&bar_a, nseg & 1);
          umma_commit(&bar_acc);
        }
        g0 += n_ct;
      }
    }
  } else {
    const int ew = warp - 2, quarter = warp & 3;                 // lane quarter
    const int grp = ew / (4 * CG), cg = (ew % (4 * CG)) >> 2, slot = grp * CG + cg;   // warp set, column group
    const int row = quarter * 32 + lane;
    const uint32_t lane_base = (uint32_t)(quarter * 32) << 16;
    uint32_t g0 = 0, nseg = 0;   // ring position of the segment's first tile; segment count (parity of bar_a / bar_acc)
    for (CeSeg sg = seg0; sg.valid; g0 += sg.n, ++nseg, sg.advance()) {
    const int r0 = sg.row_tile * kT, n_ct = sg.n, jg0 = sg.j0;   // first row (token or item), column tiles [jg0, jg0 + n_ct)
    const bool partial = PERSIST && n_ct != n_ct_all;            // other CTAs hold the rest of this row tile's columns
    float crow = 0.f;
    if (MODE == 0) crow = (r0 + row < n_valid) ? cvec[r0 + row] : -INFINITY;
    if (FUSED) crow = (r0 + row < n_valid) ? (direct.use_lse_off ? -direct.lse[r0 + row] * kLog2e : 0.f) : -INFINITY;
    float zacc = 0.f;  // FUSED: sum of G~ over this thread's columns (BCE: of softplus)
    float gsum = 0.f;  // COL mode with bias: sum over tokens of G (before the e^{b_i} row factor) -> bias gradient
    // BCE, COL mode: the item's bias enters every logit of the row (rows beyond the catalog are never written)
    const float brow = (BCE && COLCONST && HAS_BIAS && r0 + row < n_items) ? bias[r0 + row] : 0.f;
    if (A_TMEM) {
      // thread (row, column group) copies its slice of the row tile from global memory into TMEM: K elements
      // [cg*D/CG, (cg+1)*D/CG) of row r0+row -> packed columns [cg*D/(2CG), ...); rows beyond the matrix read as zero
      constexpr int WORDS = D / 2 / kSlots;  // 32-bit words per thread
      static_assert(WORDS % 16 == 0, "row-tile copy works in 16-word TMEM stores");
      const bool in = (r0 + row) < n_rows;
      const uint4* src = reinterpret_cast<const uint4*>(a_rows + (size_t)(in ? r0 + row : 0) * D + slot * (D / kSlots));
#pragma unroll
      for (int c = 0; c < WORDS; c += 16) {
        uint32_t v[16];
#pragma unroll
        for (int q = 0; q < 16; q += 4) {
          const uint4 t4 = in ? __ldg(src + ((c + q) >> 2)) : make_uint4(0u, 0u, 0u, 0u);
          v[q] = t4.x; v[q + 1] = t4.y; v[q + 2] = t4.z; v[q + 3] = t4.w;
        }
        if (PRESCALE) {   // fused pass: the row tile carries log2(e), so S comes out of the tensor core in log2 units
#pragma unroll
          for (int q = 0; q < 16; ++q) {
            const float2 f = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&v[q]));
            v[q] = pack_bf16(f.x * kLog2e, f.y * kLog2e);
          }
        }
        tmem_st16(tmem_a + lane_base + slot * WORDS + c, v);
      }
      tmem_st_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&bar_a);
    }
    // Software pipeline over CW-column chunks of this warp's kW = 64 columns: while the exponentials of one chunk run, the
    // tcgen05.ld of the next chunk of the SAME tile is in flight.  A warp-wide load occupies the quarter's TMEM read port for
    // ~2 cycles per column (256 cycles per tile and SM sub-partition); with load-everything -> wait -> compute that time was
    // MUFU idle time (ncu r2b: MUFU 61-65 % busy, ~1400 cycles per tile against 1024 of MUFU work and 1168 of tensor work).
    // The pipeline does NOT reach into the next tile: S of tile j+1 only completes one tile of tensor work after the G of tile
    // j-1 was handed over (two S buffers, in-order issue), i.e. about when this tile's epilogue ends - a prefetch placed
    // before this tile's last chunk waited ~500 cycles for it (measured r2i: 1.02 -> 1.44 ms).
    constexpr int CW = 16, NCH = kW / CW;
    static_assert(NCH >= 2 && NCH % 2 == 0, "chunk pipeline: pairs of 16-column chunks");
    // the first chunk of the NEXT tile is fetched before this tile's last chunk is exponentiated - only with >= 3 S buffers:
    // with two, S of tile j+1 completes about when the epilogue of tile j ends (measured r2i: such a prefetch costs 40 %)
    // (a set's next tile is j + GROUPS; its S is issued behind the second GEMM of tile j + GROUPS - NBUF, which must not
    //  depend on THIS tile's G: NBUF > GROUPS)
    constexpr bool PREFETCH = (NBUF >= 3) && (NBUF > GROUPS);
    auto s_wait = [&](int j) {   // j: tile of this segment; g0 + j: its position in the S-buffer / smem rings
      mbar_wait(&bar_sfull[(g0 + j) % NSTAGE], ((g0 + j) / NSTAGE) & 1);
      tc_fence_after();
    };
    auto s_addr = [&](int j) -> uint32_t { return tmem + lane_base + (uint32_t)((g0 + j) % NBUF) * TN + cg * kW; };
    uint32_t rawA[CW], rawB[CW];
#if RP_CE_ABLATE == 4
#pragma unroll
    for (int q = 0; q < CW; ++q) rawA[q] = rawB[q] = __float_as_uint(-1.f - 0.01f * (lane + q));
#endif
    for (int j = grp; j < n_ct; j += GROUPS) {   // two warp sets: this one owns every GROUPS-th column tile (= one S buffer)
      const uint32_t b = (g0 + j) % NBUF, s = (g0 + j) % NSTAGE;
      if (COLCONST) mbar_wait(&bar_full[s], ((g0 + j) / NSTAGE) & 1);  // s_cc[s] was written by the async proxy
      if (threadIdx.x == 64) RP_CTR(0, g0 + j);   // epilogue arrives at tile
      if (!PREFETCH || j == grp || RP_CE_ABLATE == 2) s_wait(j);
      if (threadIdx.x == 64) RP_CTR(1, g0 + j);   // S observed complete
#if RP_CE_ABLATE == 2  // diagnostic build (tools/ce_variants.sh): no epilogue work at all -> MMA + TMA pipeline alone
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&bar_pfull[b]);
      continue;
#endif
      const uint32_t sbase = s_addr(j);
      // G = exp2(S*log2e + offset) of one CW-column chunk -> CW/2 packed bf16 pairs, written in place over the warp's own
      // (already consumed) S columns: chunk k lands in packed columns [k CW/2, (k+1) CW/2)
      auto chunk_e = [&](const uint32_t (&raw)[CW], int k, auto every_c) {
        constexpr int EVERY = decltype(every_c)::value;
        uint32_t pk[CW / 2];
        const int col0 = (jg0 + j) * TN + cg * kW + k * CW;
        if (COLCONST && BCE) {
          const float4* cc = reinterpret_cast<const float4*>(&s_cc[s][cg * kW + k * CW]);
#pragma unroll
          for (int q = 0; q < CW; q += 4) {
            const float4 o = cc[q >> 2];   // 0 (valid token) or -inf
            const float g0_ = bce_sigmoid(__uint_as_float(raw[q + 0]) + brow + o.x);
            const float g1_ = bce_sigmoid(__uint_as_float(raw[q + 1]) + brow + o.y);
            const float g2_ = bce_sigmoid(__uint_as_float(raw[q + 2]) + brow + o.z);
            const float g3_ = bce_sigmoid(__uint_as_float(raw[q + 3]) + brow + o.w);
            if (HAS_BIAS) gsum += (g0_ + g1_) + (g2_ + g3_);
            pk[(q >> 1) + 0] = pack_bf16(g0_, g1_);
            pk[(q >> 1) + 1] = pack_bf16(g2_, g3_);
          }
        } else if (COLCONST) {
          const float4* cc = reinterpret_cast<const float4*>(&s_cc[s][cg * kW + k * CW]);
#pragma unroll
          for (int q = 0; q < CW; q += 4) {
            const float4 o = cc[q >> 2];
            const float g0_ = ce_ex2<3, EVERY>(fmaf(__uint_as_float(raw[q + 0]), kLog2e, o.x), q + 0);
            const float g1_ = ce_ex2<3, EVERY>(fmaf(__uint_as_float(raw[q + 1]), kLog2e, o.y), q + 1);
            const float g2_ = ce_ex2<3, EVERY>(fmaf(__uint_as_float(raw[q + 2]), kLog2e, o.z), q + 2);
            const float g3_ = ce_ex2<3, EVERY>(fmaf(__uint_as_float(raw[q + 3]), kLog2e, o.w), q + 3);
            if (HAS_BIAS) gsum += (g0_ + g1_) + (g2_ + g3_);
            pk[(q >> 1) + 0] = pack_bf16(g0_, g1_);
            pk[(q >> 1) + 1] = pack_bf16(g2_, g3_);
          }
        } else {
          float sv[CW];
#pragma unroll
          for (int q = 0; q < CW; ++q) sv[q] = __uint_as_float(raw[q]);
          if (HAS_BIAS) {  // per-column bias: s + b before the exponential (warp-uniform 16-byte loads)
#pragma unroll
            for (int q = 0; q < CW; q += 4) {
              const float4 b4 = __ldg(reinterpret_cast<const float4*>(bias + col0 + q));
              sv[q + 0] += b4.x;
              sv[q + 1] += b4.y;
              sv[q + 2] += b4.z;
              sv[q + 3] += b4.w;
            }
          }
          if (BCE) {
            if (col0 + CW > n_items) {  // (warp-uniform) ragged last tile: the missing items' zero rows would give s = b_i
#pragma unroll
              for (int q = 0; q < CW; ++q)
                if (col0 + q >= n_items) sv[q] = -INFINITY;
            }
            float z0 = 0.f, z1 = 0.f;
#pragma unroll
            for (int q = 0; q < CW; q += 2) {
              float sp0, sp1;
              const float g0_ = bce_terms(sv[q + 0], sp0);
              const float g1_ = bce_terms(sv[q + 1], sp1);
              z0 += sp0;
              z1 += sp1;
              pk[q >> 1] = pack_bf16(g0_, g1_);
            }
            zacc += z0 + z1;
          } else if (col0 + CW <= n_items) {  // (warp-uniform) every column of this chunk exists: no per-element masking in the hot loop
            float z0 = 0.f, z1 = 0.f;
#pragma unroll
            for (int q = 0; q < CW; q += 2) {
              const float g0_ = PRESCALE ? ce_ex2<3, EVERY>(sv[q + 0], q + 0) : ce_ex2<3, EVERY>(fmaf(sv[q + 0], kLog2e, crow), q + 0);
              const float g1_ = PRESCALE ? ce_ex2<3, EVERY>(sv[q + 1], q + 1) : ce_ex2<3, EVERY>(fmaf(sv[q + 1], kLog2e, crow), q + 1);
              if (FUSED) {
                z0 += g0_;
                z1 += g1_;
              }
              pk[q >> 1] = pack_bf16(g0_, g1_);
            }
            if (FUSED) zacc += z0 + z1;
          } else {  // ragged last tile of the catalog: columns beyond it do not exist
#pragma unroll
            for (int q = 0; q < CW; q += 2) {
              float g0_ = PRESCALE ? ex2f(sv[q + 0]) : ex2f(fmaf(sv[q + 0], kLog2e, crow));
              float g1_ = PRESCALE ? ex2f(sv[q + 1]) : ex2f(fmaf(sv[q + 1], kLog2e, crow));
              if (col0 + q >= n_items) g0_ = 0.f;
              if (col0 + q + 1 >= n_items) g1_ = 0.f;
              if (FUSED) zacc += g0_ + g1_;
              pk[q >> 1] = pack_bf16(g0_, g1_);
            }
          }
        }
#if RP_CE_ABLATE == 1  // diagnostic build: keep the TMEM traffic, drop the exponentials (G = bf16(S))
#pragma unroll
        for (int q = 0; q < CW; q += 2) pk[q >> 1] = pack_bf16(__uint_as_float(raw[q]), __uint_as_float(raw[q + 1]));
#endif
#if RP_CE_ABLATE == 3   // diagnostic: exponentials without the TMEM store of G
        if (pk[0] == 0x12345678u && pk[CW / 2 - 1] == 0x9abcdef0u) tmem_st8(sbase + k * (CW / 2), pk);
#else
        tmem_st8(sbase + k * (CW / 2), pk);
#endif
      };
      // the two epilogue warps that share the MMA-issuing thread's sub-partition (lane quarter 1) lose ~700 cycles per tile to
      // its blocked dispatch: RP_CE_POLY_EVERY_Q1 moves a share of THEIR exponentials to the FMA pipe
      auto chunk = [&](const uint32_t (&raw)[CW], int k) {
        if (RP_CE_POLY_EVERY_Q1 != RP_CE_POLY_EVERY_BWD && quarter == 1)
          chunk_e(raw, k, std::integral_constant<int, RP_CE_POLY_EVERY_Q1>{});
        else
          chunk_e(raw, k, std::integral_constant<int, RP_CE_POLY_EVERY_BWD>{});
      };
#if RP_CE_ABLATE == 4   // diagnostic: no TMEM loads (the exponentials run on whatever the registers hold)
#define tmem_ld16(a, r) asm volatile("" : "+r"(r[0]), "+r"(r[5]), "+r"(r[10]), "+r"(r[15]))
#endif
      if (!PREFETCH || j == grp) tmem_ld16(sbase, rawA);
#pragma unroll
      for (int k = 0; k < NCH; k += 2) {
        tmem_ld_wait();                                   // chunk k has landed in rawA
        tmem_ld16(sbase + (k + 1) * CW, rawB);            // chunk k+1 is on its way while chunk k is exponentiated
        chunk(rawA, k);
        tmem_ld_wait();                                   // chunk k+1 has landed in rawB
        if (k + 2 < NCH) {
          tmem_ld16(sbase + (k + 2) * CW, rawA);
        } else if (PREFETCH && j + GROUPS < n_ct) {       // S of the set's next tile was issued long ago: normally complete
          s_wait(j + GROUPS);
          tmem_ld16(s_addr(j + GROUPS), rawA);
        }
        chunk(rawB, k + 1);
      }
#if RP_CE_ABLATE == 4
#undef tmem_ld16
#endif
      if (threadIdx.x == 64) RP_CTR(2, g0 + j);   // exponentials done, stores issued
      tmem_st_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&bar_pfull[b]);
      if (threadIdx.x == 64) RP_CTR(3, g0 + j);   // G handed to the MMA thread
      if (lane == 0) RP_CTR(8 + (ew & 7), g0 + j);
    }
    // ---- final: accumulator -> global; this warp owns accumulator columns [cg*D/CG, (cg+1)*D/CG), 16 at a time
    mbar_wait(&bar_acc, nseg & 1);
    tc_fence_after();
    const int r = r0 + row;
    constexpr int DW = D / kSlots;
    const uint32_t abase = tmem_acc + lane_base + slot * DW;
    if (COLCONST) {
      float* o = reinterpret_cast<float*>(out);
      // biased head: G carries a per-item factor e^{b_i}; it was left out of the loop and is applied to the row here
      // (BCE: G carries no such factor, the 1 / T_v of the mean is applied here)
      const float rs = BCE ? loss_inv[0] : ((HAS_BIAS && r < n_items) ? __expf(bias[r]) : 1.f);
      if (HAS_BIAS) {
        s_gsum[slot][row] = gsum;
        asm volatile("bar.sync 1, %0;" ::"r"(kEW * 32) : "memory");  // epilogue warps only
        if (slot == 0 && r < n_items) {
          float tot = 0.f;
#pragma unroll
          for (int k = 0; k < kSlots; ++k) tot += s_gsum[k][row];
          if (partial) atomicAdd(d_bias + r, tot * rs); else d_bias[r] = tot * rs;
        }
        if (PERSIST) asm volatile("bar.sync 1, %0;" ::"r"(kEW * 32) : "memory");  // s_gsum is rewritten by the next segment
      }
#pragma unroll 1
      for (int c = 0; c < DW; c += 16) {
        uint32_t a16[16];
        tmem_ld16(abase + c, a16);
        tmem_ld_wait();
        if (r < n_items) {
          float4* dst = reinterpret_cast<float4*>(o + (size_t)r * D + slot * DW + c);
#pragma unroll
          for (int q = 0; q < 16; q += 4) {
            const float4 v = make_float4(__uint_as_float(a16[q]) * rs, __uint_as_float(a16[q + 1]) * rs,
                                         __uint_as_float(a16[q + 2]) * rs, __uint_as_float(a16[q + 3]) * rs);
            // a slice of the row tile's columns: 16-byte vector reduction into the zeroed output (at most two CTAs share a
            // row tile while a CTA's slice is longer than one row tile's column range, so the sum does not depend on order)
            if (partial) atomicAdd(dst + (q >> 2), v); else dst[q >> 2] = v;
          }
        }
      }
      // the accumulator / row-tile columns are handed back to the MMA thread by the next segment's bar_a arrivals
      tc_fence_before();
    } else if (FUSED && direct.d_hc != nullptr) {
      // ---- no column splits: finish here.  z_t = sum of the four slots' row sums; dH = acc / (z T_v) - E[y] / T_v
      s_gsum[slot][row] = zacc;
      asm volatile("bar.sync 1, %0;" ::"r"(kEW * 32) : "memory");
      float z = 0.f;
#pragma unroll
      for (int k = 0; k < kSlots; ++k) z += s_gsum[k][row];
      const bool live = r < n_valid;
      const float inv_n = n_valid > 0 ? 1.f / (float)n_valid : 0.f;
      const int y = live ? labels[r] : 0;
      float wg = (live && direct.row.w_ext) ? direct.row.w_ext[r] : 1.f;   // gradient weight of the row
      if (!BCE && direct.row.kind == 1) {
        // LogInCE: the weight needs the target logit before the gradient can be scaled - one extra pass over h . E[y]
        float dp = 0.f;
        if (live) {
          const uint4* ey = reinterpret_cast<const uint4*>(table + (size_t)y * D + slot * DW);
          const uint4* hr = reinterpret_cast<const uint4*>(a_rows + (size_t)r * D + slot * DW);
#pragma unroll
          for (int q = 0; q < DW / 8; ++q) {
            const uint4 e = __ldg(ey + q), hh = __ldg(hr + q);
            const __nv_bfloat162* e2 = reinterpret_cast<const __nv_bfloat162*>(&e);
            const __nv_bfloat162* h2 = reinterpret_cast<const __nv_bfloat162*>(&hh);
#pragma unroll
            for (int pp = 0; pp < 4; ++pp) {
              const float2 ef = __bfloat1622float2(e2[pp]), hf = __bfloat1622float2(h2[pp]);
              dp = fmaf(hf.x, ef.x, fmaf(hf.y, ef.y, dp));
            }
          }
        }
        s_dot[slot][row] = dp;
        asm volatile("bar.sync 1, %0;" ::"r"(kEW * 32) : "memory");
        float zy0 = 0.f;
#pragma unroll
        for (int k = 0; k < kSlots; ++k) zy0 += s_dot[k][row];
        if (HAS_BIAS) zy0 += bias[y];
        asm volatile("bar.sync 1, %0;" ::"r"(kEW * 32) : "memory");   // s_dot is written again below
        float rl_unused;
        if (live) ce_row_terms(direct.row, r, __logf(z) - crow * kLn2, zy0, rl_unused, wg);
      }
      const float scale = live ? (BCE ? inv_n : wg * inv_n / z) : 0.f;   // BCE: G is final, no normaliser
      const float lab = BCE ? inv_n : wg * inv_n;
      float dot = 0.f;
#pragma unroll 1
      for (int c = 0; c < DW; c += 16) {
        uint32_t a16[16];
        tmem_ld16(abase + c, a16);
        tmem_ld_wait();
        if (live) {
          const uint4* ey = reinterpret_cast<const uint4*>(table + (size_t)y * D + slot * DW + c);
          const uint4* hr = reinterpret_cast<const uint4*>(a_rows + (size_t)r * D + slot * DW + c);
          uint4* dst = reinterpret_cast<uint4*>(direct.d_hc + (size_t)r * D + slot * DW + c);
#pragma unroll
          for (int q = 0; q < 16; q += 8) {
            const uint4 e = __ldg(ey + (q >> 3)), hh = __ldg(hr + (q >> 3));
            const __nv_bfloat162* e2 = reinterpret_cast<const __nv_bfloat162*>(&e);
            const __nv_bfloat162* h2 = reinterpret_cast<const __nv_bfloat162*>(&hh);
            uint4 w;
            uint32_t* w32 = reinterpret_cast<uint32_t*>(&w);
#pragma unroll
            for (int pp = 0; pp < 4; ++pp) {
              const float2 ef = __bfloat1622float2(e2[pp]), hf = __bfloat1622float2(h2[pp]);
              dot = fmaf(hf.x, ef.x, fmaf(hf.y, ef.y, dot));
              w32[pp] = pack_bf16(__uint_as_float(a16[q + 2 * pp]) * scale - lab * ef.x,
                                  __uint_as_float(a16[q + 2 * pp + 1]) * scale - lab * ef.y);
            }
            dst[q >> 3] = w;
          }
        }
      }
      s_dot[slot][row] = dot;
      asm volatile("bar.sync 1, %0;" ::"r"(kEW * 32) : "memory");
      if (slot == 0 && r < capacity) {
        if (live) {
          float zy = 0.f;
#pragma unroll
          for (int k = 0; k < kSlots; ++k) zy += s_dot[k][row];
          if (HAS_BIAS) zy += bias[y];
          if (BCE) {   // row loss: sum_i softplus(s_i) - s_y (the dE pass's token mask is written by the loss reduction)
            direct.row_loss[r] = z - zy;
          } else {
          const float lse2 = log2f(z) - crow;   // (crow = 0 unless the pass runs behind the two-pass forward)
          float rl, wg2;
          ce_row_terms(direct.row, r, lse2 * kLn2, zy, rl, wg2);
          direct.lse[r] = lse2 * kLn2;
          direct.cvec[r] = -lse2 + log2f(wg2 * inv_n);
          direct.row_loss[r] = rl;
          if (direct.row.roww) direct.row.roww[r] = wg2;
          }
        } else if (!BCE) {
          direct.cvec[r] = -INFINITY;  // rows beyond T_v contribute nothing to the dE pass
        }
      }
    } else if (FUSED) {
      // partial (this column split) un-normalised gradient and row sums; ce_fused_finalize_kernel reduces the splits
      float* o = reinterpret_cast<float*>(out) + (size_t)split * capacity * D;
      if (r < n_valid) zpart[((size_t)split * kSlots + slot) * capacity + r] = zacc;
#pragma unroll 1
      for (int c = 0; c < DW; c += 16) {
        uint32_t a16[16];
        tmem_ld16(abase + c, a16);
        tmem_ld_wait();
        if (r < n_valid) {
          float4* dst = reinterpret_cast<float4*>(o + (size_t)r * D + slot * DW + c);
#pragma unroll
          for (int q = 0; q < 16; q += 4)
            dst[q >> 2] = make_float4(__uint_as_float(a16[q]), __uint_as_float(a16[q + 1]), __uint_as_float(a16[q + 2]),
                                      __uint_as_float(a16[q + 3]));
        }
      }
    } else {
      __nv_bfloat16* o = reinterpret_cast<__nv_bfloat16*>(out);
      const float inv_n = loss_inv[0] * ((direct.row.roww && r < n_valid) ? direct.row.roww[r] : 1.f);
      const int y = (r < n_valid) ? labels[r] : 0;
#pragma unroll 1
      for (int c = 0; c < DW; c += 16) {
        uint32_t a16[16];
        tmem_ld16(abase + c, a16);
        tmem_ld_wait();
        if (r < n_valid) {
          const uint4* ey = reinterpret_cast<const uint4*>(table + (size_t)y * D + slot * DW + c);
          uint4* dst = reinterpret_cast<uint4*>(o + (size_t)r * D + slot * DW + c);
#pragma unroll
          for (int q = 0; q < 16; q += 8) {
            const uint4 e = ey[q >> 3];
            const __nv_bfloat162* e2 = reinterpret_cast<const __nv_bfloat162*>(&e);
            uint4 w;
            uint32_t* w32 = reinterpret_cast<uint32_t*>(&w);
#pragma unroll
            for (int p = 0; p < 4; ++p) {
              const float2 ef = __bfloat1622float2(e2[p]);
              w32[p] = pack_bf16(__uint_as_float(a16[q + 2 * p]) - inv_n * ef.x,
                                 __uint_as_float(a16[q + 2 * p + 1]) - inv_n * ef.y);
            }
            dst[q >> 3] = w;
          }
        }
      }
    }
    }  // segments
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem, 512);
}

// dE[y_t, :] -= Hc[t, :] / T_v   (fp32 atomics; several tokens may share a label)
__global__ void ce_label_scatter_kernel(const __nv_bfloat16* __restrict__ hc, const int32_t* __restrict__ labels,
                                        const float* __restrict__ loss_inv, const int32_t* __restrict__ n_valid_ptr,
                                        int d, float* __restrict__ dE, float* __restrict__ d_bias,
                                        const float* __restrict__ roww) {
  const int n_valid = *n_valid_ptr;
  const float inv_n0 = loss_inv[0];
  if (d_bias)
    for (int t = blockIdx.x * blockDim.x + threadIdx.x; t < n_valid; t += gridDim.x * blockDim.x)
      atomicAdd(d_bias + labels[t], -inv_n0 * (roww ? roww[t] : 1.f));
  const int per_row = d / 4;   // one 16-byte vector reduction (red.global.add.v4.f32) per 4 columns
  const long long total = (long long)n_valid * per_row;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int t = (int)(i / per_row), c = (int)(i % per_row) * 4;
    const float inv_n = inv_n0 * (roww ? roww[t] : 1.f);
    const uint2 raw = *reinterpret_cast<const uint2*>(hc + (size_t)t * d + c);
    const float2 h0 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&raw.x));
    const float2 h1 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&raw.y));
    atomicAdd(reinterpret_cast<float4*>(dE + (size_t)labels[t] * d + c),
              make_float4(-inv_n * h0.x, -inv_n * h0.y, -inv_n * h1.x, -inv_n * h1.y));
  }
}

// ---- safety bound of the fused (single-reference-max) path: |s_ti + b_i| <= max_t||h_t|| * max_i||e_i|| + max|b|
__global__ void ce_bound_kernel(const __nv_bfloat16* __restrict__ hc, const __nv_bfloat16* __restrict__ table,
                                const float* __restrict__ bias, const int32_t* __restrict__ n_valid_ptr, int n_items, int d,
                                unsigned int* __restrict__ bound /* [3] float bits, zeroed */) {
  // G = min(32, d/8) lanes share one row with 16-byte loads (d/8 chunks per row, d in {64,128,256,512}); every thread keeps
  // 4 rows in flight, so the 20 MB of operands stream instead of waiting on one shuffle chain per row.
  const int n_valid = *n_valid_ptr;
  const int lane = threadIdx.x & 31;
  const int cpr = d >> 3, G = cpr < 32 ? cpr : 32, per_lane = cpr / G;     // chunks per row / lanes per row / chunks per lane
  const int rows_per_warp = 32 / G;
  const int sub = lane / G, gl = lane % G;
  const long long warp_id = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const long long n_warps = (long long)gridDim.x * (blockDim.x >> 5);
  const int total = n_valid + n_items;
  float mh = 0.f, me = 0.f, mb = 0.f;
  for (long long r0 = warp_id * rows_per_warp * 4; r0 < total; r0 += n_warps * rows_per_warp * 4) {
    float ss[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const long long r = r0 + u * rows_per_warp + sub;
      if (r < total) {
        const __nv_bfloat16* row = r < n_valid ? hc + (size_t)r * d : table + (size_t)(r - n_valid) * d;
        for (int k = 0; k < per_lane; ++k) {
          const uint4 v = __ldg(reinterpret_cast<const uint4*>(row) + gl + k * G);
          const __nv_bfloat162* h2 = reinterpret_cast<const __nv_bfloat162*>(&v);
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const float2 f = __bfloat1622float2(h2[q]);
            ss[u] = fmaf(f.x, f.x, fmaf(f.y, f.y, ss[u]));
          }
        }
      }
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      for (int o = G >> 1; o > 0; o >>= 1) ss[u] += __shfl_xor_sync(0xffffffffu, ss[u], o);
      const long long r = r0 + u * rows_per_warp + sub;
      if (r < total) {
        if (r < n_valid) mh = fmaxf(mh, ss[u]); else me = fmaxf(me, ss[u]);
        if (r >= n_valid && bias && gl == 0) mb = fmaxf(mb, fabsf(bias[r - n_valid]));
      }
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    mh = fmaxf(mh, __shfl_xor_sync(0xffffffffu, mh, o));
    me = fmaxf(me, __shfl_xor_sync(0xffffffffu, me, o));
    mb = fmaxf(mb, __shfl_xor_sync(0xffffffffu, mb, o));
  }
  if (lane == 0) {  // non-negative floats order like their bit patterns
    atomicMax(bound + 0, __float_as_uint(mh));
    atomicMax(bound + 1, __float_as_uint(me));
    atomicMax(bound + 2, __float_as_uint(mb));
  }
}

__global__ void ce_flag_kernel(const unsigned int* __restrict__ bound, int32_t* __restrict__ safe_flag) {
  const float b = sqrtf(__uint_as_float(bound[0]) * __uint_as_float(bound[1])) + __uint_as_float(bound[2]);
  // exp2(b * log2e) and its reciprocal must stay far inside the fp32 / bf16 exponent range
  *safe_flag = (b * kLog2e < 100.f) ? 1 : 0;
}

// reduce the column splits of the fused pass: lse, loss, exponent offsets for the dE pass, and
//   dHc[t] = sum_p dH~_p[t] / (z_t * T_v) - E[y_t] / T_v
__global__ void ce_fused_finalize_kernel(const float* __restrict__ part_dh, const float* __restrict__ zpart,
                                         const __nv_bfloat16* __restrict__ hc, const __nv_bfloat16* __restrict__ table,
                                         const int32_t* __restrict__ labels, const float* __restrict__ bias,
                                         const int32_t* __restrict__ n_valid_ptr, const int32_t* __restrict__ safe_flag,
                                         int n_splits, int z_slots, int capacity, int d, float* __restrict__ lse_out,
                                         float* __restrict__ cvec, __nv_bfloat16* __restrict__ d_hc,
                                         float* __restrict__ block_sums, unsigned int* __restrict__ ticket,
                                         float* __restrict__ loss_out, const CeRowOpts row, int use_lse_off, int run_if_safe) {
  if ((*safe_flag != 0) != (run_if_safe != 0)) return;
  const int n_valid = *n_valid_ptr;
  const float inv_n = n_valid > 0 ? 1.f / (float)n_valid : 0.f;
  const int lane = threadIdx.x & 31, wpb = blockDim.x >> 5;
  float local = 0.f;
  for (int t = blockIdx.x * wpb + (threadIdx.x >> 5); t < capacity; t += gridDim.x * wpb) {
    if (t >= n_valid) {
      if (lane == 0) cvec[t] = -INFINITY;
      continue;
    }
    float z = 0.f;
    for (int i = lane; i < n_splits * z_slots; i += 32) z += zpart[(size_t)i * capacity + t];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) z += __shfl_xor_sync(0xffffffffu, z, o);
    const int y = labels[t];
    const __nv_bfloat16* hr = hc + (size_t)t * d;
    const __nv_bfloat16* er = table + (size_t)y * d;
    // target logit first: the per-row variants (CeRowOpts) scale the gradient with a weight that may depend on it
    float dot = 0.f;
    for (int c = lane * 4; c < d; c += 128) {
      const uint2 hraw = *reinterpret_cast<const uint2*>(hr + c), eraw = *reinterpret_cast<const uint2*>(er + c);
      const float2 h0 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&hraw.x));
      const float2 h1 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&hraw.y));
      const float2 e0 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&eraw.x));
      const float2 e1 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&eraw.y));
      dot = fmaf(h0.x, e0.x, fmaf(h0.y, e0.y, fmaf(h1.x, e1.x, fmaf(h1.y, e1.y, dot))));
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) dot += __shfl_xor_sync(0xffffffffu, dot, o);
    if (bias) dot += bias[y];
    const float lse2 = log2f(z) + (use_lse_off ? lse_out[t] * kLog2e : 0.f);   // behind the two-pass forward: offsets -lse
    float rl, wg;
    ce_row_terms(row, t, lse2 * kLn2, dot, rl, wg);
    const float scale = wg * inv_n / z, lab = wg * inv_n;
    for (int c = lane * 4; c < d; c += 128) {  // 16-byte loads of the partials, all splits in flight
      const uint2 eraw = *reinterpret_cast<const uint2*>(er + c);
      const float2 e0 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&eraw.x));
      const float2 e1 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&eraw.y));
      float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll 8
      for (int p = 0; p < n_splits; ++p) {
        const float4 v = __ldg(reinterpret_cast<const float4*>(part_dh + ((size_t)p * capacity + t) * d + c));
        a.x += v.x; a.y += v.y; a.z += v.z; a.w += v.w;
      }
      uint2 o;
      o.x = pack_bf16(a.x * scale - lab * e0.x, a.y * scale - lab * e0.y);
      o.y = pack_bf16(a.z * scale - lab * e1.x, a.w * scale - lab * e1.y);
      *reinterpret_cast<uint2*>(d_hc + (size_t)t * d + c) = o;
    }
    if (lane == 0) {
      lse_out[t] = lse2 * kLn2;
      cvec[t] = -lse2 + log2f(wg * inv_n);
      if (row.roww) row.roww[t] = wg;
      local += rl;
    }
  }
  __shared__ float red[32];
  __shared__ bool last;
  if (lane == 0) red[threadIdx.x >> 5] = local;
  __syncthreads();
  if (threadIdx.x == 0) {
    float sum = 0.f;
    for (int i = 0; i < wpb; ++i) sum += red[i];
    block_sums[blockIdx.x] = sum;
    __threadfence();
    last = (atomicAdd(ticket, 1u) == gridDim.x - 1);
  }
  __syncthreads();
  if (last && threadIdx.x == 0) {
    __threadfence();
    float sum = 0.f;
    for (int i = 0; i < (int)gridDim.x; ++i) sum += reinterpret_cast<volatile float*>(block_sums)[i];
    loss_out[0] = sum * inv_n;
    loss_out[1] = inv_n;
  }
}

// d = 512 path: dH[c0 + r, :] = sum_s part[s][r, :] - E[y, :] / T_v   (split-K partials of softmax . E / T_v; the one-hot
// part of softmax - onehot is subtracted here), rows c0 + r < *n_valid.  One warp per row.
__global__ void ce_dh_reduce_kernel(const float* __restrict__ part, int n_splits, long long split_stride, int rows, int c0,
                                    __nv_bfloat16* __restrict__ d_hc, const __nv_bfloat16* __restrict__ table,
                                    const int32_t* __restrict__ labels, const float* __restrict__ loss_inv,
                                    const int32_t* __restrict__ n_valid_ptr, int d, const float* __restrict__ roww) {
  const int n_valid = *n_valid_ptr;
  const int lane = threadIdx.x & 31, wpb = blockDim.x >> 5;
  for (int r = blockIdx.x * wpb + (threadIdx.x >> 5); r < rows && c0 + r < n_valid; r += gridDim.x * wpb) {
    const int t = c0 + r;
    const float inv_n = loss_inv[0] * (roww ? roww[t] : 1.f);
    const __nv_bfloat16* e = table + (size_t)labels[t] * d;
    for (int c = lane * 4; c < d; c += 128) {
      float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
      for (int sp = 0; sp < n_splits; ++sp) {
        const float4 v = *reinterpret_cast<const float4*>(part + (size_t)sp * split_stride + (size_t)r * d + c);
        a.x += v.x; a.y += v.y; a.z += v.z; a.w += v.w;
      }
      const uint2 ev = *reinterpret_cast<const uint2*>(e + c);
      const float2 e0 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&ev.x));
      const float2 e1 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&ev.y));
      uint2 o;
      o.x = pack_bf16(a.x - inv_n * e0.x, a.y - inv_n * e0.y);
      o.y = pack_bf16(a.z - inv_n * e1.x, a.w - inv_n * e1.y);
      *reinterpret_cast<uint2*>(d_hc + (size_t)t * d + c) = o;
    }
  }
}

// d = 512: S and the [128 x 512] fp32 gradient accumulator do not fit the 512 TMEM columns together, so the backward
// materialises the softmax numerators G (bf16) for a chunk of tokens at a time and runs three plain GEMMs per chunk.
// Chunk rows: as many as fit the G budget (RP_CE_WIDE_G_BYTES, default 8 GiB), multiple of 128.
static long long wide_ldg(int n_items) { return ((long long)n_items + 63) / 64 * 64; }
static int wide_chunk_rows(int cap, int n_items) {
  const char* env = getenv("RP_CE_WIDE_G_BYTES");  // read per call: the workspace query and the launch must agree
  const long long budget = env ? atoll(env) : (8ll << 30);
  long long rows = budget / (wide_ldg(n_items) * 2) / 128 * 128;
  const long long cap128 = ((long long)cap + 127) / 128 * 128;
  if (rows < 128) rows = 128;
  if (rows > cap128) rows = cap128;
  return (int)rows;
}

// ---- full-catalog BCE head: completion of the fused pass
// n_splits == 1 (the fused kernel wrote dH and the row losses): mean loss over the valid targets in a fixed order, 1 / T_v,
// and the dE pass's token mask (0 for t < T_v, -inf up to the padded capacity)
__global__ void __launch_bounds__(1024) bce_loss_reduce_kernel(const float* __restrict__ row_loss,
                                                               const int32_t* __restrict__ n_valid_ptr, int cap128,
                                                               float* __restrict__ mask, float* __restrict__ loss_out) {
  __shared__ float red[1024];
  const int n_valid = *n_valid_ptr;
  float a = 0.f;
  for (int i = threadIdx.x; i < n_valid; i += 1024) a += row_loss[i];
  for (int i = threadIdx.x; i < cap128; i += 1024) mask[i] = i < n_valid ? 0.f : -INFINITY;
  red[threadIdx.x] = a;
  __syncthreads();
  for (int o = 512; o > 0; o >>= 1) {
    if ((int)threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    const float inv_n = n_valid > 0 ? 1.f / (float)n_valid : 0.f;
    loss_out[0] = red[0] * inv_n;
    loss_out[1] = inv_n;
  }
}

// n_splits > 1: reduce the column splits.  One warp per token:  dHc[t] = (sum_p dH~_p[t] - E[y_t]) / T_v,
// row loss = sum of the softplus partials - s_y (fp32 gather-dot, + b_y); the token mask as above; deterministic loss sum
// (per-block partials, the last block adds them in index order)
__global__ void bce_finalize_kernel(const float* __restrict__ part_dh, const float* __restrict__ zpart,
                                    const __nv_bfloat16* __restrict__ hc, const __nv_bfloat16* __restrict__ table,
                                    const int32_t* __restrict__ labels, const float* __restrict__ bias,
                                    const int32_t* __restrict__ n_valid_ptr, int n_splits, int z_slots, int capacity, int cap128,
                                    int d, __nv_bfloat16* __restrict__ d_hc, float* __restrict__ mask,
                                    float* __restrict__ block_sums, unsigned int* __restrict__ ticket,
                                    float* __restrict__ loss_out) {
  const int n_valid = *n_valid_ptr;
  const float inv_n = n_valid > 0 ? 1.f / (float)n_valid : 0.f;
  const int lane = threadIdx.x & 31, wpb = blockDim.x >> 5;
  float local = 0.f;
  for (int t = blockIdx.x * wpb + (threadIdx.x >> 5); t < cap128; t += gridDim.x * wpb) {
    if (t >= n_valid || t >= capacity) {
      if (lane == 0) mask[t] = -INFINITY;
      continue;
    }
    float z = 0.f;
    for (int i = lane; i < n_splits * z_slots; i += 32) z += zpart[(size_t)i * capacity + t];
    const int y = labels[t];
    const __nv_bfloat16* hr = hc + (size_t)t * d;
    const __nv_bfloat16* er = table + (size_t)y * d;
    float dot = 0.f;
    for (int c = lane * 4; c < d; c += 128) {
      const uint2 hraw = *reinterpret_cast<const uint2*>(hr + c), eraw = *reinterpret_cast<const uint2*>(er + c);
      const float2 h0 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&hraw.x));
      const float2 h1 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&hraw.y));
      const float2 e0 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&eraw.x));
      const float2 e1 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&eraw.y));
      dot = fmaf(h0.x, e0.x, fmaf(h0.y, e0.y, fmaf(h1.x, e1.x, fmaf(h1.y, e1.y, dot))));
      float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll 8
      for (int p = 0; p < n_splits; ++p) {
        const float4 v = __ldg(reinterpret_cast<const float4*>(part_dh + ((size_t)p * capacity + t) * d + c));
        a.x += v.x; a.y += v.y; a.z += v.z; a.w += v.w;
      }
      uint2 o;
      o.x = pack_bf16((a.x - e0.x) * inv_n, (a.y - e0.y) * inv_n);
      o.y = pack_bf16((a.z - e1.x) * inv_n, (a.w - e1.y) * inv_n);
      *reinterpret_cast<uint2*>(d_hc + (size_t)t * d + c) = o;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      z += __shfl_xor_sync(0xffffffffu, z, o);
      dot += __shfl_xor_sync(0xffffffffu, dot, o);
    }
    if (bias) dot += bias[y];
    if (lane == 0) {
      mask[t] = 0.f;
      local += z - dot;
    }
  }
  __shared__ float red[32];
  __shared__ bool last;
  if (lane == 0) red[threadIdx.x >> 5] = local;
  __syncthreads();
  if (threadIdx.x == 0) {
    float sum = 0.f;
    for (int i = 0; i < wpb; ++i) sum += red[i];
    block_sums[blockIdx.x] = sum;
    __threadfence();
    last = (atomicAdd(ticket, 1u) == gridDim.x - 1);
  }
  __syncthreads();
  if (last && threadIdx.x == 0) {
    __threadfence();
    float sum = 0.f;
    for (int i = 0; i < (int)gridDim.x; ++i) sum += reinterpret_cast<volatile float*>(block_sums)[i];
    loss_out[0] = sum * inv_n;
    loss_out[1] = inv_n;
  }
}

static int pick_splits(int n_row_tiles, int n_col_tiles, int max_splits = 8) {
  const int sms = sm_count();
  int best = 1;
  double best_eff = 0.0;
  for (int p = 1; p <= max_splits && p <= n_col_tiles; ++p) {
    const long long ctas = (long long)n_row_tiles * p;
    const double eff = (double)ctas / (double)(((ctas + sms - 1) / sms) * sms);
    if (eff > best_eff + 0.02) {
      best_eff = eff;
      best = p;
    }
  }
  return best;
}

}  // namespace rp

using namespace rp;

// workspace layout: [part float2 cap*8*2][block_sums 1024 f][ticket, bound[3], flag, pad -> 64 B][zpart 16*cap f]
//                   [part_dh 8*cap*d f]
struct CeWs {
  float2* part; float* block_sums; unsigned int* ticket; unsigned int* bound; int32_t* flag; float* zpart; float* roww; float* part_dh;
};
static const int kMaxSplits = 8;       // fused forward + dH: partial gradients per split
static const int kMaxSplitsFwd = 32;   // two-pass forward: only (max, sum) pairs per split
static const int kWideSplitK = 16;     // d = 512 backward: split-K partials of the dH GEMM

static size_t ce_ws_base_bytes(int cap, int d) {
  return (size_t)cap * kMaxSplitsFwd * 2 * sizeof(float2) + 4096 + 64 + (size_t)kMaxSplits * kBwdCG * kCeMaxGroups * cap * 4 +
         (size_t)(cap + 3) / 4 * 16 + (d <= 256 ? (size_t)kMaxSplits * cap * d * 4 : 0) + 256;
}
static size_t ce_ws_bytes(int cap, int n_items, int d) {
  size_t b = (ce_ws_base_bytes(cap, d) + 1023) / 1024 * 1024;
  if (d > 256) {
    const size_t rows = (size_t)wide_chunk_rows(cap, n_items);
    b += rows * wide_ldg(n_items) * 2;              // G chunk (bf16)
    b += (size_t)kWideSplitK * rows * d * 4;        // split-K partials of dH (fp32)
  }
  return b;
}
static CeWs ce_ws(void* workspace, int cap, int d) {
  uint8_t* w = reinterpret_cast<uint8_t*>(workspace);
  CeWs r;
  r.part = reinterpret_cast<float2*>(w);
  w += (size_t)cap * kMaxSplitsFwd * 2 * sizeof(float2);
  r.block_sums = reinterpret_cast<float*>(w);
  w += 4096;
  r.ticket = reinterpret_cast<unsigned int*>(w);
  r.bound = r.ticket + 1;
  r.flag = reinterpret_cast<int32_t*>(r.ticket + 4);
  w += 64;
  r.zpart = reinterpret_cast<float*>(w);
  w += (size_t)kMaxSplits * kBwdCG * kCeMaxGroups * cap * 4;
  r.roww = reinterpret_cast<float*>(w);   // gradient weight per row (CeRowOpts), written by every forward finalisation
  w += (size_t)(cap + 3) / 4 * 16;
  r.part_dh = reinterpret_cast<float*>(w);
  (void)d;
  return r;
}

#ifdef RP_CE_TRACE
RP_API int rp_debug_ce_trace(unsigned long long* host_out, int n_words) {
  RP_CUDA_CHECK(cudaDeviceSynchronize());
  RP_CUDA_CHECK(cudaMemcpyFromSymbol(host_out, rp::g_ce_trace, sizeof(unsigned long long) * (size_t)n_words));
  return RP_OK;
}
#endif

RP_API size_t rp_ce_head_workspace(int capacity_tokens, int n_items, int d) {
  if (capacity_tokens <= 0 || n_items <= 0 || d <= 0) return 0;
  return ce_ws_bytes(capacity_tokens, n_items, d);
}

template <int KCH, int NSTAGE>
static int launch_ce_fwd(const CUtensorMap& tmA, const CUtensorMap& tmB, const int32_t* n_valid, int n_items,
                         int n_splits, int n_tok_tiles, const float* bias, float2* part, const int32_t* skip,
                         cudaStream_t stream) {
  const int smem = (KCH + NSTAGE) * kChunk + 1024;
  auto kern = ce_fwd_kernel<KCH, NSTAGE>;
  RP_CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  kern<<<n_tok_tiles * n_splits, kThreads, smem, stream>>>(tmA, tmB, n_valid, n_items, n_splits, bias, part, skip);
  RP_LAUNCH_CHECK();
  return RP_OK;
}

// two epilogue warp sets: d = 128 with two S buffers (the row-tile copy and the accumulator read-out split 4 ways there)
constexpr int ce_groups_of(int kch, int nbuf) { return (RP_CE_GROUPS == 2 && kch == 2 && nbuf == 2) ? 2 : 1; }
static int ce_z_slots(int d) {
  constexpr bool a_tmem = (RP_CE_A_TMEM != 0) && (RP_CE_ORDER == 1);
  const int nbuf = (d <= 128 && a_tmem) ? 2 : ((RP_CE_NBUF3 && d <= 128) ? 3 : 2);
  if (d <= 128 && a_tmem && RP_CE_TN64 != 0) return RP_CE_TN64_GROUPS == 2 ? 2 : kBwdCG;
  return kBwdCG * ce_groups_of(d / 64, nbuf);
}

template <int KCH, int NSTAGE, int MODE, bool BCE = false>
static int launch_ce_bwd(const CUtensorMap& tmA, const void* b_mat, int b_rows, const void* a_rows, const float* cvec,
                         const int32_t* labels,
                         const void* table, const float* loss_inv, const int32_t* n_valid, int n_items, const float* bias,
                         float* d_bias, void* out, int grid, const int32_t* safe_flag, int run_if_safe, int n_splits,
                         int capacity, float* zpart, cudaStream_t stream, const CeDirect& direct = CeDirect{nullptr, nullptr, nullptr, nullptr, CeRowOpts{nullptr, nullptr, 0, 0.f, 0.f}, 0}) {
  // d <= 128: the row tile goes to TMEM (2 S buffers + accumulator + operand = 448 columns) and its 32 KB of smem become
  // an extra pipeline stage; d = 256: row tile in smem, 2 S buffers + accumulator = 512 columns
  // RP_CE_ORDER 1: both directions keep the row tile in TMEM (two S buffers suffice once the issue order no longer drains the
  // pipe); otherwise round 1's choice (measured then: the TMEM row tile paid for the dE pass only, because it forces 2 buffers)
  constexpr bool A_TMEM = (RP_CE_A_TMEM != 0) && KCH <= 2 && (MODE == 1 || RP_CE_ORDER == 1);
  // column tiles: 64 wide in four S buffers when the row tile is in TMEM and the issue order is the in-order one (see the
  // kernel's header comment), else 128 wide in two (three without the TMEM row tile)
  constexpr int TN = (A_TMEM && RP_CE_ORDER == 1 && RP_CE_TN64 != 0) ? 64 : 128;
  constexpr int NBUF = TN == 64 ? 4 : (A_TMEM ? 2 : ((RP_CE_NBUF3 && KCH <= 2) ? 3 : 2));
  constexpr bool INORDER = (RP_CE_ORDER == 1) && (NBUF == 2 || TN == 64);
  constexpr int NST = (NSTAGE + (A_TMEM ? 1 : 0)) * (128 / TN);   // the same bytes of column tiles in flight
  const int smem = (A_TMEM ? 0 : 1) * KCH * kChunk + NST * KCH * TN * 128 + 1024;
  CUtensorMap tmB;   // column-side matrix, one [TN rows x 64 columns] box per chunk
  {
    const int rc = make_tmap_bf16(&tmB, b_mat, b_rows, KCH * 64, KCH * 64, TN);
    if (rc != RP_OK) return rc;
  }
  // the biased head (BERT4Rec) is a separate instantiation: its per-column adds / row sums cost an instruction per logit
  constexpr int GROUPS = TN == 64 ? RP_CE_TN64_GROUPS : ce_groups_of(KCH, NBUF);
  constexpr int CG = (TN == 64 && GROUPS == 2) ? 1 : kBwdCG;
  // dE pass with the row tile in TMEM: persistent work slices (see CeSeg) - `grid` row tiles become one CTA per SM, the
  // output is zeroed first because slices that end inside a row tile add their part with reductions
  constexpr bool PERSIST = (MODE == 1) && A_TMEM && (RP_CE_PERSIST != 0);
  constexpr int NI = (INORDER && RP_CE_ISSUERS > 1) ? RP_CE_ISSUERS : 1;
  auto kern = bias ? ce_bwd_kernel<KCH, NST, MODE, NBUF, A_TMEM, INORDER, true, GROUPS, PERSIST, TN, CG, NI, BCE>
                   : ce_bwd_kernel<KCH, NST, MODE, NBUF, A_TMEM, INORDER, false, GROUPS, PERSIST, TN, CG, NI, BCE>;
  RP_CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  if (PERSIST) {
    RP_CUDA_CHECK(cudaMemsetAsync(out, 0, (size_t)n_items * KCH * 64 * sizeof(float), stream));
    if (d_bias) RP_CUDA_CHECK(cudaMemsetAsync(d_bias, 0, (size_t)n_items * sizeof(float), stream));
    if (grid > sm_count()) grid = sm_count();
  }
  kern<<<grid, 64 + GROUPS * 4 * CG * 32 + (NI - 1) * 32, smem, stream>>>(tmA, tmB, reinterpret_cast<const __nv_bfloat16*>(a_rows), cvec, labels,
                                            reinterpret_cast<const __nv_bfloat16*>(table), loss_inv,
                                         n_valid, n_items, bias, d_bias, out, safe_flag, run_if_safe, n_splits, capacity, zpart, direct);
  RP_LAUNCH_CHECK();
  return RP_OK;
}

template <int MODE, bool BCE = false>
static int dispatch_ce_bwd(int d, const CUtensorMap& tmA, const void* b_mat, int b_rows, const void* a_rows, const float* cvec,
                           const int32_t* labels,
                           const void* table, const float* loss_inv, const int32_t* n_valid, int n_items, const float* bias,
                           float* d_bias, void* out, int grid, const int32_t* safe_flag, int run_if_safe, int n_splits,
                           int capacity, float* zpart, cudaStream_t stream, const CeDirect& direct = CeDirect{nullptr, nullptr, nullptr, nullptr, CeRowOpts{nullptr, nullptr, 0, 0.f, 0.f}, 0}) {
  switch (d) {
    case 64:
      return launch_ce_bwd<1, 6, MODE, BCE>(tmA, b_mat, b_rows, a_rows, cvec, labels, table, loss_inv, n_valid, n_items, bias, d_bias, out, grid,
                                       safe_flag, run_if_safe, n_splits, capacity, zpart, stream, direct);
    case 128:
      return launch_ce_bwd<2, RP_CE_NSTAGE_D128, MODE, BCE>(tmA, b_mat, b_rows, a_rows, cvec, labels, table, loss_inv, n_valid, n_items, bias, d_bias, out, grid,
                                       safe_flag, run_if_safe, n_splits, capacity, zpart, stream, direct);
    case 256:
      return launch_ce_bwd<4, 2, MODE, BCE>(tmA, b_mat, b_rows, a_rows, cvec, labels, table, loss_inv, n_valid, n_items, bias, d_bias, out, grid,
                                       safe_flag, run_if_safe, n_splits, capacity, zpart, stream, direct);
    default:
      return RP_ESHAPE;
  }
}

// Forward of the CE head.  hc bf16 [capacity, d] (rows >= *n_valid ignored), table bf16 [n_items, d], labels int32
// [capacity], n_valid int32 [1] (device).  Outputs: loss_out fp32 [2] = {mean CE, 1/T_v}; lse fp32 [capacity]; cvec fp32
// (exponent offsets consumed by rp_ce_head_bwd).
// d_hc != NULL (training, d <= 256) enables the FUSED path: one pass computes the row sums of exp(s) against a fixed
// reference maximum of 0 together with the un-normalised gradient sum_i exp(s_i) E_i, so the separate log-sum-exp pass
// disappears and d_hc is already final after this call.  A device-side Cauchy-Schwarz bound on |s| guards the trick; if
// it fails the two-pass kernels run instead (both variants are launched, the losing one exits at once), so the call
// stays CUDA-graph capturable.  n_valid_hint (host estimate of *n_valid, 0 = unknown) only tunes the load balance.
RP_API int rp_ce_head_fwd_w(const void* hc, const void* table, const float* bias, const int32_t* labels,
                            const int32_t* n_valid, int capacity, int n_items, int d, float* loss_out, float* lse, float* cvec,
                            void* d_hc, int n_valid_hint, const float* row_weight, int loss_kind, float log_eps, float clamp,
                            void* workspace, size_t workspace_bytes, void* stream_);
RP_API int rp_ce_head_fwd(const void* hc, const void* table, const float* bias, const int32_t* labels,
                          const int32_t* n_valid, int capacity, int n_items, int d, float* loss_out, float* lse, float* cvec,
                          void* d_hc, int n_valid_hint, void* workspace, size_t workspace_bytes, void* stream_) {
  return rp_ce_head_fwd_w(hc, table, bias, labels, n_valid, capacity, n_items, d, loss_out, lse, cvec, d_hc, n_valid_hint, nullptr,
                          0, 0.f, 0.f, workspace, workspace_bytes, stream_);
}

// Per-row variants of the head (CeRowOpts): row_weight fp32 [capacity] (>= 0, compacted order of the valid targets, NULL = 1),
// loss_kind 0 = CE, 1 = LogInCE with (log_eps, clamp).  The backward must be rp_ce_head_bwd with the SAME workspace (the
// per-row gradient weights live there); everything else as rp_ce_head_fwd.
RP_API int rp_ce_head_fwd_w(const void* hc, const void* table, const float* bias, const int32_t* labels,
                            const int32_t* n_valid, int capacity, int n_items, int d, float* loss_out, float* lse, float* cvec,
                            void* d_hc, int n_valid_hint, const float* row_weight, int loss_kind, float log_eps, float clamp,
                            void* workspace, size_t workspace_bytes, void* stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  if (loss_kind != 0 && loss_kind != 1) return RP_EINVAL;
  if (!hc || !table || !labels || !n_valid || !loss_out || !lse || !cvec || !workspace) return RP_EINVAL;
  if (capacity <= 0 || n_items <= 0) return RP_ESHAPE;
  if (d != 64 && d != 128 && d != 256 && d != 512) return RP_ESHAPE;
  if (workspace_bytes < ce_ws_bytes(capacity, n_items, d)) return RP_EWORKSPACE;
  const bool fused = d_hc != nullptr && d <= 256;
  const int n_tok_tiles = (capacity + kT - 1) / kT, n_item_tiles = (n_items + kT - 1) / kT;
  const int hint_tiles = (n_valid_hint > 0 && n_valid_hint <= capacity) ? (n_valid_hint + kT - 1) / kT : n_tok_tiles;
  CeWs ws = ce_ws(workspace, capacity, d);
  CUtensorMap tmA, tmB;
  int rc;
  if ((rc = make_tmap_bf16(&tmA, hc, capacity, d, d, 128)) != RP_OK) return rc;
  if ((rc = make_tmap_bf16(&tmB, table, n_items, d, d, 128)) != RP_OK) return rc;
  RP_CUDA_CHECK(cudaMemsetAsync(ws.ticket, 0, 64, stream));  // ticket, bound[3], flag
  const int32_t* skip = nullptr;
  int blocks = (capacity + 7) / 8;
  if (blocks > 1024) blocks = 1024;
  if (fused) {
    ce_bound_kernel<<<sm_count() * 8, 256, 0, stream>>>(reinterpret_cast<const __nv_bfloat16*>(hc),
                                                        reinterpret_cast<const __nv_bfloat16*>(table), bias, n_valid, n_items, d,
                                                        ws.bound);
    RP_LAUNCH_CHECK();
    ce_flag_kernel<<<1, 1, 0, stream>>>(ws.bound, ws.flag);
    RP_LAUNCH_CHECK();
    const int P = pick_splits(hint_tiles, n_item_tiles);
    CeDirect direct{nullptr, lse, nullptr, nullptr, CeRowOpts{row_weight, ws.roww, loss_kind, log_eps, clamp}, 0};
    if (P == 1) {  // every CTA sees the whole catalog: lse / dH / loss terms come straight out of the fused kernel
      direct.d_hc = reinterpret_cast<__nv_bfloat16*>(d_hc);
      direct.cvec = cvec;
      direct.row_loss = ws.zpart;  // the row-sum partials are not needed in this mode: reuse their buffer
    }
    rc = dispatch_ce_bwd<2>(d, tmA, table, n_items, hc, cvec, labels, table, loss_out + 1, n_valid, n_items, bias, nullptr, ws.part_dh,
                            n_tok_tiles * P, ws.flag, 1, P, capacity, ws.zpart, stream, direct);
    if (rc != RP_OK) return rc;
    if (P == 1) {
      ce_loss_reduce_kernel<<<1, 1024, 0, stream>>>(ws.zpart, n_valid, ws.flag, loss_out, 1);
      RP_LAUNCH_CHECK();
    } else
    ce_fused_finalize_kernel<<<blocks, 256, 0, stream>>>(ws.part_dh, ws.zpart, reinterpret_cast<const __nv_bfloat16*>(hc),
                                                         reinterpret_cast<const __nv_bfloat16*>(table), labels, bias, n_valid,
                                                         ws.flag, P, ce_z_slots(d), capacity, d, lse, cvec,
                                                         reinterpret_cast<__nv_bfloat16*>(d_hc), ws.block_sums, ws.ticket, loss_out,
                                                         CeRowOpts{row_weight, ws.roww, loss_kind, log_eps, clamp}, 0, 1);
    RP_LAUNCH_CHECK();
    skip = ws.flag;
  }
  int P2 = pick_splits(hint_tiles, n_item_tiles, kMaxSplitsFwd);
  if (fused) {  // two-pass fallback behind the fused pass: it only runs when the bound failed; launching (and retiring) tens of
                // thousands of CTAs that exit at once cost ~40 us per step, so keep it at about two waves
    const int cap = (2 * sm_count() + n_tok_tiles - 1) / n_tok_tiles;
    if (P2 > cap) P2 = cap;
  }
  switch (d) {
    case 64: rc = launch_ce_fwd<1, 8>(tmA, tmB, n_valid, n_items, P2, n_tok_tiles, bias, ws.part, skip, stream); break;
    case 128: rc = launch_ce_fwd<2, 8>(tmA, tmB, n_valid, n_items, P2, n_tok_tiles, bias, ws.part, skip, stream); break;
    case 256: rc = launch_ce_fwd<4, 8>(tmA, tmB, n_valid, n_items, P2, n_tok_tiles, bias, ws.part, skip, stream); break;
    default: rc = launch_ce_fwd<8, 5>(tmA, tmB, n_valid, n_items, P2, n_tok_tiles, bias, ws.part, skip, stream); break;
  }
  if (rc != RP_OK) return rc;
  ce_finalize_kernel<<<blocks, 256, 0, stream>>>(ws.part, reinterpret_cast<const __nv_bfloat16*>(hc),
                                                 reinterpret_cast<const __nv_bfloat16*>(table), labels, bias, n_valid, P2 * 2,
                                                 capacity, d, lse, cvec, ws.block_sums, ws.ticket, loss_out, skip,
                                                 CeRowOpts{row_weight, ws.roww, loss_kind, log_eps, clamp});
  RP_LAUNCH_CHECK();
  if (fused) {
    // The bound failed (these launches exit at once otherwise): the two-pass forward above has produced lse; the gradient
    // dH comes from the SAME fused kernel, now with the exponent offset -lse[t] per row (G = softmax, z ~ 1) - with its column
    // splits and all SMs busy, where the row-tile-per-CTA MODE 0 pass ran 32 CTAs at BERT4Rec's ~4000 masked positions
    // (2.2 ms of a 4.3 ms step at config 3, whose un-normalised outputs outgrow the bound within a few hundred steps).
    const int P = pick_splits(hint_tiles, n_item_tiles);
    CeDirect direct{nullptr, lse, nullptr, nullptr, CeRowOpts{row_weight, ws.roww, loss_kind, log_eps, clamp}, 1};
    if (P == 1) {
      direct.d_hc = reinterpret_cast<__nv_bfloat16*>(d_hc);
      direct.cvec = cvec;
      direct.row_loss = ws.zpart;
    }
    RP_CUDA_CHECK(cudaMemsetAsync(ws.ticket, 0, 4, stream));   // the deterministic loss reduction's ticket was used above
    rc = dispatch_ce_bwd<2>(d, tmA, table, n_items, hc, cvec, labels, table, loss_out + 1, n_valid, n_items, bias, nullptr, ws.part_dh,
                            n_tok_tiles * P, ws.flag, 0, P, capacity, ws.zpart, stream, direct);
    if (rc != RP_OK) return rc;
    if (P == 1) {
      ce_loss_reduce_kernel<<<1, 1024, 0, stream>>>(ws.zpart, n_valid, ws.flag, loss_out, 0);
    } else {
      ce_fused_finalize_kernel<<<blocks, 256, 0, stream>>>(ws.part_dh, ws.zpart, reinterpret_cast<const __nv_bfloat16*>(hc),
                                                           reinterpret_cast<const __nv_bfloat16*>(table), labels, bias, n_valid,
                                                           ws.flag, P, ce_z_slots(d), capacity, d, lse, cvec,
                                                           reinterpret_cast<__nv_bfloat16*>(d_hc), ws.block_sums, ws.ticket, loss_out,
                                                           CeRowOpts{row_weight, ws.roww, loss_kind, log_eps, clamp}, 1, 0);
    }
    RP_LAUNCH_CHECK();
  }
  return RP_OK;
}

// Backward of rp_ce_head_fwd for d(loss) = 1:
//   d_hc   bf16 [capacity, d]  (rows < *n_valid) - already written by the forward when it ran fused (`fused` != 0 and the
//          device-side bound held); otherwise computed here from the stored lse.  d = 512: chunked materialised-G path
//          (three GEMMs per token chunk, see wide_chunk_rows), workspace required
//   d_table fp32 [n_items, d]  OVERWRITTEN with softmax^T . hc / T_v, then the one-hot part is atomically subtracted
//   d_bias  fp32 [n_items] (iff bias)  OVERWRITTEN likewise.        d in {64,128,256}; 512 without bias.
RP_API int rp_ce_head_bwd(const void* hc, const void* table, const float* bias, const int32_t* labels,
                          const int32_t* n_valid, int capacity, int n_items, int d, const float* loss_out /* from fwd */,
                          const float* cvec /* from fwd */, void* d_hc, float* d_table, float* d_bias, int fused,
                          int n_valid_hint, void* workspace, size_t workspace_bytes, void* stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  if (!hc || !table || !labels || !n_valid || !loss_out || !cvec || !d_hc || !d_table) return RP_EINVAL;
  if ((bias == nullptr) != (d_bias == nullptr)) return RP_EINVAL;
  if (capacity <= 0 || n_items <= 0) return RP_ESHAPE;
  if (d != 64 && d != 128 && d != 256 && d != 512) return RP_ESHAPE;
  if ((fused || d == 512) && (!workspace || workspace_bytes < ce_ws_bytes(capacity, n_items, d))) return RP_EWORKSPACE;
  // gradient weight per row, written by the forward (all ones for the plain CE head); without a workspace: plain head
  const float* roww = (workspace && workspace_bytes >= ce_ws_bytes(capacity, n_items, d)) ? ce_ws(workspace, capacity, d).roww : nullptr;
  if (d == 512) {
    // ---- wide-hidden path: per token chunk  G = exp2((hc.E^T + b) log2e + c_t)  ->  dH = G.E,  dE += G^T.hc
    if (bias) return RP_ESHAPE;  // biased (BERT4Rec) head at d = 512 is not built
    const long long ldg = wide_ldg(n_items);
    const int chunk = wide_chunk_rows(capacity, n_items);
    uint8_t* G = reinterpret_cast<uint8_t*>(workspace) + (ce_ws_base_bytes(capacity, d) + 1023) / 1024 * 1024;
    float* part = reinterpret_cast<float*>(G + (size_t)chunk * ldg * 2);
    const long long part_stride = (long long)chunk * d;
    const int hint = (n_valid_hint > 0 && n_valid_hint < capacity) ? n_valid_hint : capacity;
    int rc;
    for (int c0 = 0, it = 0; c0 < capacity; c0 += chunk, ++it) {
      const int rows = (capacity - c0 < chunk) ? capacity - c0 : chunk;
      rp_gemm_desc g;
      memset(&g, 0, sizeof(g));
      g.batch = 1; g.inner = 1; g.alpha = 1.f; g.split_k = 1;
      // G [rows, n_items] = exp2((hc[c0:c0+rows] . E^T) log2e + cvec)
      g.A = reinterpret_cast<const __nv_bfloat16*>(hc) + (size_t)c0 * d; g.a_rows = rows; g.a_cols = d; g.lda = d; g.a_mn = 0;
      g.B = table; g.b_rows = n_items; g.b_cols = d; g.ldb = d; g.b_mn = 0;
      g.M = rows; g.N = n_items; g.K = d;
      g.C = G; g.ldc = ldg; g.out_mode = 0; g.act = 3; g.row_exp2_offset = cvec + c0;
      g.m_limit_dev = n_valid; g.m_limit_base = c0;
      if ((rc = rp_gemm(&g, stream_)) != RP_OK) return rc;
      // dH[c0:c0+rows] = G . E - onehot   (A = G K-major over the items, B = E read MN-major).  Few row tiles against a
      // contraction over the whole catalog: split-K partials (fp32, deterministic), reduced together with the label term
      int live = hint - c0;
      live = live < 128 ? 128 : (live > rows ? rows : live);
      int split = (2 * sm_count()) / (((live + 127) / 128) * (d / 128));
      split = split < 1 ? 1 : (split > kWideSplitK ? kWideSplitK : split);
      memset(&g, 0, sizeof(g));
      g.batch = 1; g.inner = 1; g.alpha = 1.f; g.split_k = split;
      g.A = G; g.a_rows = rows; g.a_cols = n_items; g.lda = ldg; g.a_mn = 0;
      g.B = table; g.b_rows = n_items; g.b_cols = d; g.ldb = d; g.b_mn = 1;
      g.M = rows; g.N = d; g.K = n_items;
      g.C = part; g.ldc = d; g.out_mode = 3; g.c_split_stride = part_stride;
      g.m_limit_dev = n_valid; g.m_limit_base = c0;
      if ((rc = rp_gemm(&g, stream_)) != RP_OK) return rc;
      ce_dh_reduce_kernel<<<sm_count() * 4, 256, 0, stream>>>(part, split, part_stride, rows, c0,
                                                               reinterpret_cast<__nv_bfloat16*>(d_hc),
                                                               reinterpret_cast<const __nv_bfloat16*>(table), labels,
                                                               loss_out + 1, n_valid, d, roww);
      RP_LAUNCH_CHECK();
      // dE (+)= G^T . hc[c0:c0+rows]      (A = G read MN-major, contraction over the chunk's valid tokens)
      memset(&g, 0, sizeof(g));
      g.batch = 1; g.inner = 1; g.alpha = 1.f; g.split_k = 1;
      g.A = G; g.a_rows = rows; g.a_cols = n_items; g.lda = ldg; g.a_mn = 1;
      g.B = reinterpret_cast<const __nv_bfloat16*>(hc) + (size_t)c0 * d; g.b_rows = rows; g.b_cols = d; g.ldb = d; g.b_mn = 1;
      g.M = n_items; g.N = d; g.K = rows;
      g.C = d_table; g.ldc = d; g.out_mode = it == 0 ? 2 : 4;
      g.k_limit_dev = n_valid; g.k_limit_base = c0;
      if ((rc = rp_gemm(&g, stream_)) != RP_OK) return rc;
    }
    ce_label_scatter_kernel<<<sm_count() * 4, 256, 0, stream>>>(reinterpret_cast<const __nv_bfloat16*>(hc), labels, loss_out + 1,
                                                                 n_valid, d, d_table, d_bias, roww);
    RP_LAUNCH_CHECK();
    return RP_OK;
  }
  CUtensorMap tmH, tmE;
  int rc;
  if ((rc = make_tmap_bf16(&tmH, hc, capacity, d, d, 128)) != RP_OK) return rc;
  if ((rc = make_tmap_bf16(&tmE, table, n_items, d, d, 128)) != RP_OK) return rc;
  const int n_tok_tiles = (capacity + kT - 1) / kT, n_item_tiles = (n_items + kT - 1) / kT;
  const float* loss_inv = loss_out + 1;
  const int32_t* flag = fused ? ce_ws(workspace, capacity, d).flag : nullptr;
  // token-major pass: only when the forward did not already produce d_hc (a fused forward always does: from the fused pass
  // itself, or - bound failed - from its second launch behind the two-pass forward)
  if (!fused)
  rc = dispatch_ce_bwd<0>(d, tmH, table, n_items, hc, cvec, labels, table, loss_inv, n_valid, n_items, bias, nullptr, d_hc, n_tok_tiles, flag, 0,
                          1, capacity, nullptr, stream,
                          CeDirect{nullptr, nullptr, nullptr, nullptr, CeRowOpts{nullptr, const_cast<float*>(roww), 0, 0.f, 0.f}});
  if (rc != RP_OK) return rc;
  rc = dispatch_ce_bwd<1>(d, tmE, hc, capacity, table, cvec, labels, table, loss_inv, n_valid, n_items, bias, d_bias, d_table, n_item_tiles,
                          nullptr, 0, 1, capacity, nullptr, stream);
  if (rc != RP_OK) return rc;
  ce_label_scatter_kernel<<<sm_count() * 4, 256, 0, stream>>>(reinterpret_cast<const __nv_bfloat16*>(hc), labels, loss_inv,
                                                               n_valid, d, d_table, d_bias, roww);
  RP_LAUNCH_CHECK();
  return RP_OK;
}

// ---------------------------------------------------------------------------------------------------------------------
// Full-catalog BCE head (BCEWithLogitsLoss(reduction="sum") / T_v against a one-hot target row): the fused forward + dH pass
// and the persistent dE pass of the CE head with the BCE epilogues (ce_bwd_kernel<..., BCE = true>).  No normaliser, so no
// lse, no bound on |s| and no two-pass fallback.
// workspace: [block_sums 1024 f][ticket, pad -> 64 B][zpart 16*cap f (also the row losses)][mask round_up(cap,128) f]
//            [part_dh 8*cap*d f]
// ---------------------------------------------------------------------------------------------------------------------
struct BceWs {
  float* block_sums; unsigned int* ticket; float* zpart; float* mask; float* part_dh;
};
static size_t bce_zpart_bytes(int cap) { return ((size_t)kMaxSplits * kBwdCG * kCeMaxGroups * cap * 4 + 255) / 256 * 256; }
static size_t bce_mask_bytes(int cap) { return ((size_t)(cap + 127) / 128 * 128 * 4 + 255) / 256 * 256; }
static size_t bce_ws_bytes(int cap, int d) {
  return 4096 + 256 + bce_zpart_bytes(cap) + bce_mask_bytes(cap) + (size_t)kMaxSplits * cap * d * 4;
}
static BceWs bce_ws(void* workspace, int cap) {
  uint8_t* w = reinterpret_cast<uint8_t*>(workspace);
  BceWs r;
  r.block_sums = reinterpret_cast<float*>(w);
  w += 4096;
  r.ticket = reinterpret_cast<unsigned int*>(w);
  w += 256;
  r.zpart = reinterpret_cast<float*>(w);
  w += bce_zpart_bytes(cap);
  r.mask = reinterpret_cast<float*>(w);
  w += bce_mask_bytes(cap);
  r.part_dh = reinterpret_cast<float*>(w);
  return r;
}

RP_API size_t rp_bce_head_workspace(int capacity_tokens, int n_items, int d) {
  if (capacity_tokens <= 0 || n_items <= 0 || (d != 64 && d != 128 && d != 256)) return 0;
  return bce_ws_bytes(capacity_tokens, d);
}

// Forward + dH.  loss_out fp32 [2] = {mean BCE over the valid targets, 1 / T_v}; d_hc bf16 [capacity, d] (rows < *n_valid)
// is final after this call.  n_valid_hint: host estimate of *n_valid (0 = unknown), load balance only.
RP_API int rp_bce_head_fwd(const void* hc, const void* table, const float* bias, const int32_t* labels, const int32_t* n_valid,
                           int capacity, int n_items, int d, float* loss_out, void* d_hc, int n_valid_hint, void* workspace,
                           size_t workspace_bytes, void* stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  if (!hc || !table || !labels || !n_valid || !loss_out || !d_hc || !workspace) return RP_EINVAL;
  if (capacity <= 0 || n_items <= 0) return RP_ESHAPE;
  if (d != 64 && d != 128 && d != 256) return RP_ESHAPE;
  if (workspace_bytes < bce_ws_bytes(capacity, d)) return RP_EWORKSPACE;
  const int n_tok_tiles = (capacity + kT - 1) / kT, n_item_tiles = (n_items + kT - 1) / kT;
  const int hint_tiles = (n_valid_hint > 0 && n_valid_hint <= capacity) ? (n_valid_hint + kT - 1) / kT : n_tok_tiles;
  BceWs ws = bce_ws(workspace, capacity);
  CUtensorMap tmA;
  int rc;
  if ((rc = make_tmap_bf16(&tmA, hc, capacity, d, d, 128)) != RP_OK) return rc;
  const int P = pick_splits(hint_tiles, n_item_tiles);
  CeDirect direct{nullptr, nullptr, nullptr, nullptr, CeRowOpts{nullptr, nullptr, 0, 0.f, 0.f}, 0};
  if (P == 1) {  // every CTA sees the whole catalog: dH and the row losses come straight out of the fused kernel
    direct.d_hc = reinterpret_cast<__nv_bfloat16*>(d_hc);
    direct.row_loss = ws.zpart;
  }
  rc = dispatch_ce_bwd<2, true>(d, tmA, table, n_items, hc, nullptr, labels, table, nullptr, n_valid, n_items, bias, nullptr,
                                ws.part_dh, n_tok_tiles * P, nullptr, 1, P, capacity, ws.zpart, stream, direct);
  if (rc != RP_OK) return rc;
  const int cap128 = n_tok_tiles * kT;
  if (P == 1) {
    bce_loss_reduce_kernel<<<1, 1024, 0, stream>>>(ws.zpart, n_valid, cap128, ws.mask, loss_out);
  } else {
    RP_CUDA_CHECK(cudaMemsetAsync(ws.ticket, 0, 4, stream));
    int blocks = (cap128 + 7) / 8;
    if (blocks > 1024) blocks = 1024;
    bce_finalize_kernel<<<blocks, 256, 0, stream>>>(ws.part_dh, ws.zpart, reinterpret_cast<const __nv_bfloat16*>(hc),
                                                    reinterpret_cast<const __nv_bfloat16*>(table), labels, bias, n_valid, P,
                                                    ce_z_slots(d), capacity, cap128, d, reinterpret_cast<__nv_bfloat16*>(d_hc),
                                                    ws.mask, ws.block_sums, ws.ticket, loss_out);
  }
  RP_LAUNCH_CHECK();
  return RP_OK;
}

// dE (and d_bias) of rp_bce_head_fwd for d(loss) = 1, with the SAME workspace and loss_out:
//   d_table fp32 [n_items, d]  OVERWRITTEN with sigmoid^T . hc / T_v, then the one-hot part is atomically subtracted
//   d_bias  fp32 [n_items] (iff bias)  OVERWRITTEN likewise
RP_API int rp_bce_head_bwd(const void* hc, const void* table, const float* bias, const int32_t* labels, const int32_t* n_valid,
                           int capacity, int n_items, int d, const float* loss_out, float* d_table, float* d_bias, void* workspace,
                           size_t workspace_bytes, void* stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  if (!hc || !table || !labels || !n_valid || !loss_out || !d_table || !workspace) return RP_EINVAL;
  if ((bias == nullptr) != (d_bias == nullptr)) return RP_EINVAL;
  if (capacity <= 0 || n_items <= 0) return RP_ESHAPE;
  if (d != 64 && d != 128 && d != 256) return RP_ESHAPE;
  if (workspace_bytes < bce_ws_bytes(capacity, d)) return RP_EWORKSPACE;
  BceWs ws = bce_ws(workspace, capacity);
  CUtensorMap tmE;
  int rc;
  if ((rc = make_tmap_bf16(&tmE, table, n_items, d, d, 128)) != RP_OK) return rc;
  const int n_item_tiles = (n_items + kT - 1) / kT;
  const float* loss_inv = loss_out + 1;
  rc = dispatch_ce_bwd<1, true>(d, tmE, hc, capacity, table, ws.mask, labels, table, loss_inv, n_valid, n_items, bias, d_bias,
                                d_table, n_item_tiles, nullptr, 0, 1, capacity, nullptr, stream);
  if (rc != RP_OK) return rc;
  ce_label_scatter_kernel<<<sm_count() * 4, 256, 0, stream>>>(reinterpret_cast<const __nv_bfloat16*>(hc), labels, loss_inv,
                                                               n_valid, d, d_table, d_bias, nullptr);
  RP_LAUNCH_CHECK();
  return RP_OK;
}
