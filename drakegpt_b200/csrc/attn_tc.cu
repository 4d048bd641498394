// Tensor-mode fused causal attention for sm_100a (head size 64, T in {128, 256}).
//
// Forward  (persistent: one CTA per SM walks a balanced list of (batch, head, 128-query tile)
//   items, two in flight):
//   TMA loads Q, K, V tiles (128B swizzle) -> tcgen05.mma S = Q K^T into TMEM (the whole
//   128 x T score row block fits: no online rescaling) -> one softmax thread per query row
//   reads S with tcgen05.ld, applies the causal mask, exp2, counter-based dropout, and
//   writes bf16 P back into TMEM (tcgen05.st, over the S columns already consumed) ->
//   tcgen05.mma O = P V with P as the TMEM A operand and V consumed MN-major from its
//   row-major shared-memory tile -> the same thread scales by 1/rowsum and stores bf16 O at
//   column h*64 (the head concat is free).
//   The T x T probabilities never touch HBM; only the log-sum-exp per row is saved.
//
// Backward (one CTA per (batch, head)): recomputes S = Q K^T and dP = dO V^T per
//   (query tile, key tile) pair on the tensor cores, 256 threads (two per query row) turn
//   them into Pd / dS (same counter-based mask as forward) in shared memory, and three more
//   MMAs accumulate dV += Pd^T dO, dK += dS^T Q, dQ += dS K in TMEM.  Every operand view
//   (K-major or MN-major, transposed or not) is a descriptor over the same row-major tiles.
#include <cuda.h>

#include "common.cuh"
#include "ptx.cuh"

namespace dgpt {

using namespace ptx;

int make_tmap_bf16_2d(CUtensorMap* map, const void* base, int64_t inner, int64_t outer, int64_t ld, int box_outer);

static constexpr int HD = 64;     // head size
static constexpr int QT = 128;    // query / key tile rows
static constexpr float kLog2e = 1.4426950408889634f;

struct AttnTcP {
  void *o, *dq, *dk, *dv;
  const void *o_in, *d_o;
  float* lse;
  int64_t o_rs, dq_rs, dk_rs, dv_rs, do_rs;
  int B, NH, T;
  float scale, inv_keep;
  uint32_t thr, site;
  uint64_t seed;
  const uint64_t* seed_dev;
};

__device__ __forceinline__ uint32_t pack_bf16(float a, float b) {
  __nv_bfloat162 v = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&v);
}

// write 32 consecutive bf16 (cols [c0, c0+32) of `row`) of a [128 x 64*n] K-major SW128 tile set
__device__ __forceinline__ void store_row32_sw128(uint8_t* tile_base, int row, int c0, const float (&v)[32]) {
  uint8_t* blk = tile_base + (c0 >> 6) * 16384 + row * 128;
  const int chunk0 = (c0 & 63) >> 3;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    uint4 w;
    w.x = pack_bf16(v[8 * j], v[8 * j + 1]);
    w.y = pack_bf16(v[8 * j + 2], v[8 * j + 3]);
    w.z = pack_bf16(v[8 * j + 4], v[8 * j + 5]);
    w.w = pack_bf16(v[8 * j + 6], v[8 * j + 7]);
    *reinterpret_cast<uint4*>(blk + (((chunk0 + j) ^ (row & 7)) << 4)) = w;
  }
}

// ===========================================================================
// forward, persistent: one CTA per SM walks a statically balanced list of (batch, head, query
// tile) items with TWO items in flight, so that the serial phases of one item (TMA latency, S MMAs, softmax, P V,
// output) are filled with the other item's work instead of idling the SM:
//   warp 8   TMA producer: Q / K and V tiles of item n into stage n & 1 (the Q / K stage is released as soon as the
//            S MMAs have read it, the V stage after P V: the loads of item n + 2 run during the softmax of item n)
//   warp 9   tcgen05 issuer + TMEM owner: S = Q K^T into TMEM slot n & 1 (256 columns each), later O = P V from
//            the bf16 P the softmax warps wrote over the consumed S columns (TS-mode MMA); issues whichever of
//            "S of the next item" / "P V of the oldest item" becomes ready first (non-blocking barrier tests)
//   warps 0-3 / 4-7   softmax warpgroup 0 / 1 (one thread per query row): items alternate between them, so one
//            group runs its exp2 / dropout / pack loop while the other waits for an MMA or stores its output
// The producer and the issuer sit on the highest warp ids: the sub-partition arbiter favours the highest eligible
// warp id, so their few, latency-critical instructions are never queued behind the softmax warps.
// ===========================================================================
static constexpr int kFwd2Threads = 320;
static constexpr int kFwd2QK = 49152;                              // Q 16 KB + K 2 x 16 KB per stage
static constexpr int kFwd2Smem = 2 * kFwd2QK + 2 * 32768 + 256 + 1024;  // + V stages, barriers, alignment slack
static constexpr int kWHeavy = 5, kWLight = 2;                     // relative cost of a 2-key-tile / 1-key-tile item

struct FwdSched {
  int nheavy, nlight;  // items with two key tiles (query tile 1) / one key tile (query tile 0, or T = 128)
  unsigned long long* probe;  // DGPT_CLOCK_PROBE stamps (or NULL)
};

__global__ void __launch_bounds__(kFwd2Threads, 1)
attn_fwd_tc2_kernel(const __grid_constant__ CUtensorMap map_q32, const __grid_constant__ CUtensorMap map_k,
                    const __grid_constant__ CUtensorMap map_v, AttnTcP p, FwdSched sc) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint8_t* sQK = smem;                    // [2][Q | K0 | K1]
  uint8_t* sV = smem + 2 * kFwd2QK;       // [2][4 x 8 KB]
  uint64_t* bars = reinterpret_cast<uint64_t*>(sV + 2 * 32768);
  uint64_t *qk_full = bars, *qk_empty = bars + 2, *v_full = bars + 4, *v_empty = bars + 6, *s_full = bars + 8,
           *p_full = bars + 10, *o_full = bars + 12, *slot_free = bars + 14;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 16);

  clock_probe_begin(sc.probe);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int ntile = p.T / QT;

  // ---- this CTA's item list (closed form, identical in every warp) ----
  // heavy items round-robin; light items fill every CTA up to the same weighted load; the few left over round-robin
  const int G = gridDim.x, c = blockIdx.x;
  const int hq = sc.nheavy / G, hr = sc.nheavy % G;
  const int nh_c = hq + (c < hr ? 1 : 0);
  const int U = (kWHeavy * sc.nheavy + kWLight * sc.nlight + G - 1) / G;
  const int cap_hi = max(0, (U - kWHeavy * (hq + 1)) / kWLight), cap_lo = max(0, (U - kWHeavy * hq) / kWLight);
  const int cap_total = hr * cap_hi + (G - hr) * cap_lo;
  const int l_start = c < hr ? c * cap_hi : hr * cap_hi + (c - hr) * cap_lo;
  const int l0 = min(sc.nlight, l_start), l1 = min(sc.nlight, l_start + (c < hr ? cap_hi : cap_lo));
  const int n_extra = cap_total < sc.nlight ? (sc.nlight - cap_total - c + G - 1) / G : 0;
  const int n_items = nh_c + (l1 - l0) + max(0, n_extra);
  // item n -> (batch * NH + head, query tile)
  auto item = [&](int n, int& bh, int& qt) {
    if (n < nh_c) {
      const int hi = c + n * G;  // heavy: query tile 1
      bh = hi; qt = ntile - 1;
    } else {
      const int m = n - nh_c;
      const int li = m < l1 - l0 ? l0 + m : cap_total + c + (m - (l1 - l0)) * G;
      bh = li; qt = 0;
    }
  };

  if (threadIdx.x == 0) {
    prefetch_tensormap(&map_q32);
    prefetch_tensormap(&map_k);
    prefetch_tensormap(&map_v);
    for (int g = 0; g < 2; ++g) {
      mbar_init(&qk_full[g], 1);
      mbar_init(&qk_empty[g], 1);
      mbar_init(&v_full[g], 1);
      mbar_init(&v_empty[g], 1);
      mbar_init(&s_full[g], 1);
      mbar_init(&p_full[g], 4);
      mbar_init(&o_full[g], 1);
      mbar_init(&slot_free[g], 4);
    }
    fence_barrier_init();
  }
  if (warp == 9) tmem_alloc<512>(tmem_slot);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  pdl_grid_sync();  // prologue done (shared memory / TMEM only); global memory from here on

  if (warp == 8) {
    // ------------------------------ TMA producer ---------------------------
    for (int n = 0; n < n_items; ++n) {
      const int g = n & 1, k = n >> 1;
      int bh, qt;
      item(n, bh, qt);
      const int nkv = qt + 1, b = bh / p.NH, h = bh % p.NH, row0 = b * p.T;
      uint8_t* q_s = sQK + g * kFwd2QK;
      uint8_t* v_s = sV + g * 32768;
      mbar_wait(&qk_empty[g], (k & 1) ^ 1);
      if (elect_one()) {
        mbar_expect_tx(&qk_full[g], 16384 * (1 + nkv));
        // warpgroup 1 takes its query tile with the four 32-row blocks in REVERSE order: causal rows near the end of
        // the tile see more keys, and a row block is pinned to the sub-partition of its TMEM lane quadrant, so
        // sub-partition q then serves block q of warpgroup 0's item and block 3 - q of warpgroup 1's (equal load)
        for (int qb = 0; qb < 4; ++qb)
          tma_load_2d(q_s + qb * 4096, &map_q32, &qk_full[g], h * HD, row0 + qt * QT + (g ? 3 - qb : qb) * 32);
        for (int j = 0; j < nkv; ++j) tma_load_2d(q_s + 16384 * (1 + j), &map_k, &qk_full[g], h * HD, row0 + j * QT);
      }
      __syncwarp();
      mbar_wait(&v_empty[g], (k & 1) ^ 1);
      if (elect_one()) {
        mbar_expect_tx(&v_full[g], 16384 * nkv);
        for (int kb = 0; kb < 2 * nkv; ++kb) tma_load_2d(v_s + kb * 8192, &map_v, &v_full[g], h * HD, row0 + kb * 64);
      }
      __syncwarp();
    }
  } else if (warp == 9) {
    // ------------------------------ MMA issuer -----------------------------
    constexpr uint32_t idesc_s = make_idesc_bf16(128, 128, 0, 0);
    constexpr uint32_t idesc_o = make_idesc_bf16(128, 64, 0, 1);
    int next_s = 0, next_pv = 0;
    while (next_pv < n_items) {
      bool progressed = false;
      if (next_s < n_items) {
        const int g = next_s & 1, k = next_s >> 1;
        // slot g is free once the epilogue of item next_s - 2 has read its output (first use: passes at once)
        if (mbar_test(&qk_full[g], k & 1) && mbar_test(&slot_free[g], (k & 1) ^ 1)) {
          tc_fence_after();
          int bh, qt;
          item(next_s, bh, qt);
          const int nkv = qt + 1;
          const uint64_t dq0 = make_smem_desc_sw128(smem_u32(sQK + g * kFwd2QK), 16, 1024);
          const uint64_t dk0 = make_smem_desc_sw128(smem_u32(sQK + g * kFwd2QK + 16384), 16, 1024);
          if (elect_one()) {
            for (int j = 0; j < nkv; ++j) {
#pragma unroll
              for (int kk = 0; kk < 4; ++kk)
                tc_mma_bf16(tmem + g * 256 + j * 128, dq0 + (uint64_t)(kk * 2), dk0 + (uint64_t)(j * 1024 + kk * 2), idesc_s, kk > 0);
            }
            tc_commit(&s_full[g]);
            tc_commit(&qk_empty[g]);  // the Q / K stage may be refilled once these MMAs have read it
          }
          __syncwarp();
          ++next_s;
          progressed = true;
        }
      }
      if (next_pv < next_s) {
        const int g = next_pv & 1, k = next_pv >> 1;
        if (mbar_test(&p_full[g], k & 1) && mbar_test(&v_full[g], k & 1)) {
          tc_fence_after();
          int bh, qt;
          item(next_pv, bh, qt);
          const int nkv = qt + 1;
          // O = P V: P (bf16 pairs, 8 TMEM columns per UMMA_K step) overlays the consumed S columns, V is read
          // MN-major from its row-major tile, O accumulates in the columns right above P
          const uint64_t dv0 = make_smem_desc_sw128(smem_u32(sV + g * 32768), 8192, 1024);
          if (elect_one()) {
            for (int kb = 0; kb < 2 * nkv; ++kb) {
#pragma unroll
              for (int kk = 0; kk < 4; ++kk)
                tc_mma_bf16_ts(tmem + g * 256 + nkv * 64, tmem + g * 256 + kb * 32 + kk * 8, dv0 + (uint64_t)(kb * 512 + kk * 128),
                               idesc_o, (kb | kk) > 0);
            }
            tc_commit(&o_full[g]);
            tc_commit(&v_empty[g]);
          }
          __syncwarp();
          ++next_pv;
          progressed = true;
        }
      }
      if (!progressed) __nanosleep(32);
    }
  } else {
    // ---------------------------- softmax + output: one thread per query row ----------
    const int g = warp >> 2;     // warpgroup = TMEM slot = shared-memory stage
    const int quad = warp & 3;
    const int rblk = g ? 3 - quad : quad;  // which 32-row block of the query tile sits in this warp's TMEM lanes
    const int row = rblk * 32 + lane;
    const uint32_t taddr = tmem + (uint32_t)(g * 256) + ((uint32_t)(quad * 32) << 16);
    uint64_t seed = p.seed;
    if (p.thr && p.seed_dev) seed += *p.seed_dev;
    const float sc2 = p.scale * kLog2e;
    for (int n = g; n < n_items; n += 2) {
      const int k = n >> 1;
      int bh, qt;
      item(n, bh, qt);
      const int nkv = qt + 1, b = bh / p.NH, h = bh % p.NH, row0 = b * p.T;
      const int qg = qt * QT + row;  // query position inside the sequence
      const int ncols = nkv * QT;
#define FTS(i) do { if (sc.probe && blockIdx.x == 0 && warp == 0 && lane == 0 && k < 3) sc.probe[4 + k * 8 + (i)] = (unsigned long long)clock64(); } while (0)
      FTS(0);
      mbar_wait(&s_full[g], k & 1);
      FTS(1);
      tc_fence_after();
      // tcgen05.ld is warp-collective: loop bounds must be warp-uniform, so the LAST row of this warp decides which
      // 32-column chunks are fully masked; chunks entirely left of the diagonal need no per-element causal test
      const int qg_max = qt * QT + rblk * 32 + 31, qg_min = qt * QT + rblk * 32;
      float mx = -INFINITY;
      for (int cc = 0; cc < ncols && cc <= qg_max; cc += 32) {
        uint32_t r[32];
        tmem_ld32(taddr + cc, r);
        tmem_ld_wait();
        if (cc + 31 <= qg_min) {
#pragma unroll
          for (int j = 0; j < 32; ++j) mx = fmaxf(mx, __uint_as_float(r[j]));
        } else {
#pragma unroll
          for (int j = 0; j < 32; ++j)
            if (cc + j <= qg) mx = fmaxf(mx, __uint_as_float(r[j]));
        }
      }
      FTS(2);
      const float msc = mx * sc2;
      float sum = 0.f;
      const uint64_t base = (((uint64_t)b * p.NH + h) * p.T + qg) * (uint64_t)p.T;
      for (int cc = 0; cc < ncols; cc += 32) {
        float e[32];
        if (cc > qg_max) {
#pragma unroll
          for (int j = 0; j < 32; ++j) e[j] = 0.f;
        } else {
          uint32_t r[32];
          tmem_ld32(taddr + cc, r);
          tmem_ld_wait();
          if (cc + 31 <= qg_min) {
#pragma unroll
            for (int j = 0; j < 32; ++j) {
              const float v = exp2f(__uint_as_float(r[j]) * sc2 - msc);
              sum += v;
              e[j] = v;
            }
          } else {
#pragma unroll
            for (int j = 0; j < 32; ++j) {
              const float v = (cc + j <= qg) ? exp2f(__uint_as_float(r[j]) * sc2 - msc) : 0.f;
              sum += v;
              e[j] = v;
            }
          }
          if (p.thr) {  // the 32 keys of this chunk are one mask group (T % 32 == 0)
            const DropGroup dg = dropout_group(seed, p.site, (base + cc) >> 5);
#pragma unroll
            for (int j = 0; j < 32; ++j)
              if (dropout_word(dg, j) < p.thr) e[j] = 0.f;
          }
        }
        // bf16 P, two keys per 32-bit TMEM column, over S columns [cc / 2, cc / 2 + 16): already consumed by this thread
        uint32_t pk[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) pk[j] = pack_bf16(e[2 * j], e[2 * j + 1]);
        tmem_st16(taddr + (cc >> 1), pk);
      }
      if (p.lse) p.lse[((int64_t)b * p.NH + h) * p.T + qg] = mx * p.scale + logf(sum);
      tmem_st_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&p_full[g]);
      FTS(3);
      // output
      mbar_wait(&o_full[g], k & 1);
      FTS(4);
      tc_fence_after();
      const float oscale = p.inv_keep / sum;
      __nv_bfloat16* orow = reinterpret_cast<__nv_bfloat16*>(p.o) + (int64_t)(row0 + qg) * p.o_rs + h * HD;
#pragma unroll
      for (int cc = 0; cc < HD; cc += 32) {
        uint32_t r[32];
        tmem_ld32(taddr + nkv * 64 + cc, r);
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          uint4 w;
          w.x = pack_bf16(__uint_as_float(r[8 * j]) * oscale, __uint_as_float(r[8 * j + 1]) * oscale);
          w.y = pack_bf16(__uint_as_float(r[8 * j + 2]) * oscale, __uint_as_float(r[8 * j + 3]) * oscale);
          w.z = pack_bf16(__uint_as_float(r[8 * j + 4]) * oscale, __uint_as_float(r[8 * j + 5]) * oscale);
          w.w = pack_bf16(__uint_as_float(r[8 * j + 6]) * oscale, __uint_as_float(r[8 * j + 7]) * oscale);
          *reinterpret_cast<uint4*>(orow + cc + 8 * j) = w;
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&slot_free[g]);  // TMEM slot g may take the S of item n + 2
      FTS(5);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 9) {
    tc_fence_after();
    tmem_dealloc<512>(tmem);
  }
  clock_probe_end(sc.probe);
}

// ===========================================================================
// backward
// ===========================================================================
#ifdef DGPT_ATTN_TS
__device__ long long g_attn_ts[64];  // phase stamps of one CTA (BTS below), printed by launch_attn_bwd_tc
#endif
static constexpr int kBwdThreads = 64 + 256;
static constexpr int kBwdSmem = 8 * 16384 + 2 * 32768 + 16384 + 2048 + 1024 + 128;

// one 32-key chunk of one query row: P, dropout, dS -> swizzled bf16 rows of the Pd / dS tiles
template <bool DIAG, bool DROP>
__device__ __forceinline__ void bwd_chunk_math(const AttnTcP& p, uint32_t lane_addr_st, uint32_t lane_addr_dp, int row, int k0,
                                               float sc, float lse2, float Dq, uint64_t seed, uint64_t base,
                                               float (&pd)[32], float (&ds)[32]) {
  uint32_t st[32], dp[32];
  tmem_ld32(lane_addr_st + k0, st);
  tmem_ld32(lane_addr_dp + k0, dp);
  tmem_ld_wait();
  DropGroup g = {0u, 0u};
  if (DROP) g = dropout_group(seed, p.site, (base + k0) >> 5);  // the chunk's 32 keys are one mask group
#pragma unroll
  for (int t = 0; t < 32; ++t) {
    float pv = exp2f(__uint_as_float(st[t]) * sc - lse2);
    if (DIAG) pv = (k0 + t) <= row ? pv : 0.f;
    float dpv = __uint_as_float(dp[t]);
    float pdv = pv;
    if (DROP) {
      const bool keep = dropout_word(g, t) >= p.thr;
      dpv = keep ? dpv * p.inv_keep : 0.f;
      pdv = keep ? pv * p.inv_keep : 0.f;
    }
    pd[t] = pdv;
    ds[t] = pv * (dpv - Dq) * p.scale;
  }
}

template <bool DROP>
__global__ void __launch_bounds__(kBwdThreads, 1)
attn_bwd_tc_kernel(const __grid_constant__ CUtensorMap map_q, const __grid_constant__ CUtensorMap map_k,
                   const __grid_constant__ CUtensorMap map_v, const __grid_constant__ CUtensorMap map_do,
                   const __grid_constant__ CUtensorMap map_o, const __grid_constant__ CUtensorMap map_dq,
                   const __grid_constant__ CUtensorMap map_dk, const __grid_constant__ CUtensorMap map_dv, AttnTcP p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* sQ = smem;                  // [2][128 x 64]
  uint8_t* sK = smem + 2 * 16384;
  uint8_t* sV = smem + 4 * 16384;
  uint8_t* sG = smem + 6 * 16384;      // dO
  uint8_t* sPd = smem + 8 * 16384;     // Pd  [128 q x 128 kv] as two K-major 64-key blocks (first: the O tiles)
  uint8_t* sDs = sPd + 32768;          // dS  (same layout)
  uint8_t* sSt = sDs + 32768;          // [128 x 64] bf16 staging tile for the dQ / dK / dV TMA stores
  float* lse_s = reinterpret_cast<float*>(sSt + 16384);  // [256]  lse * log2(e)
  float* D_s = lse_s + 256;                              // [256]  rowsum(dO * O)
  uint64_t* bars = reinterpret_cast<uint64_t*>(D_s + 256);
  uint64_t *ld_a = bars, *st_full = bars + 1, *ps_full = bars + 2, *drained = bars + 3, *acc_done = bars + 4;
  uint64_t *ld_b = bars + 5, *ld_c = bars + 6;  // loads arrive in three stages so that pair (0,0) starts after half of them
  uint64_t* acc_free = bars + 7;                // the accumulate MMAs of a pair have retired (Pd / dS tiles reusable)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 8);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
#ifdef DGPT_ATTN_TS
#define BTS(i) do { if (blockIdx.x == 0 && blockIdx.y == (gridDim.y / 2) && warp == 2 && lane == 0) g_attn_ts[i] = clock64(); } while (0)
#else
#define BTS(i) do { } while (0)
#endif
  BTS(0);
  const int h = blockIdx.x, b = blockIdx.y;
  const int ntile = p.T / QT;
  const int npair = ntile == 1 ? 1 : 3;  // (0,0) | (0,0),(1,0),(1,1)
  const int row0 = b * p.T;

  if (threadIdx.x == 0) {
    prefetch_tensormap(&map_q);
    prefetch_tensormap(&map_k);
    prefetch_tensormap(&map_v);
    prefetch_tensormap(&map_do);
    prefetch_tensormap(&map_o);
    mbar_init(ld_a, 1);
    mbar_init(ld_b, 1);
    mbar_init(ld_c, 1);
    mbar_init(st_full, 1);
    mbar_init(ps_full, 8);
    mbar_init(drained, 8);
    mbar_init(acc_done, 1);
    mbar_init(acc_free, 1);
    fence_barrier_init();
  }
  if (warp == 0) {  // the loads do not depend on TMEM: issue them before the allocation and the CTA-wide barrier
    __syncwarp();
    pdl_grid_sync();  // ... but they do read the previous kernel's output
    if (elect_one()) {
      // stage A: everything pair (0,0) needs; B: query tile 1 (pairs (1,0), (1,1)); C: key tile 1 (pair (1,1)).
      // O is only needed for D = rowsum(dO * O): O_0 lands in the Pd tile, O_1 in the store staging tile
      // (both are consumed before their first other use).
      mbar_expect_tx(ld_a, 16384 * 5);
      tma_load_2d(sG, &map_do, ld_a, h * HD, row0);
      tma_load_2d(sPd, &map_o, ld_a, h * HD, row0);
      tma_load_2d(sQ, &map_q, ld_a, h * HD, row0);
      tma_load_2d(sK, &map_k, ld_a, h * HD, row0);
      tma_load_2d(sV, &map_v, ld_a, h * HD, row0);
      if (ntile > 1) {
        mbar_expect_tx(ld_b, 16384 * 3);
        tma_load_2d(sG + 16384, &map_do, ld_b, h * HD, row0 + QT);
        tma_load_2d(sSt, &map_o, ld_b, h * HD, row0 + QT);
        tma_load_2d(sQ + 16384, &map_q, ld_b, h * HD, row0 + QT);
        mbar_expect_tx(ld_c, 16384 * 2);
        tma_load_2d(sK + 16384, &map_k, ld_c, h * HD, row0 + QT);
        tma_load_2d(sV + 16384, &map_v, ld_c, h * HD, row0 + QT);
      }
    }
  }
  if (warp == 1) tmem_alloc<512>(tmem_slot);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  constexpr uint32_t TM_ST = 0, TM_DP = 128, TM_DV = 256, TM_DK = 320, TM_DQ = 384;
  if (warp != 0) pdl_grid_sync();  // (warp 0 passed it before issuing the loads)

  if (warp == 0) {
    // (loads were issued before the TMEM allocation, see above)
  } else if (warp == 1) {
    // whole warp in uniform control flow, one elected lane issues (see forward)
    constexpr uint32_t id_kk = make_idesc_bf16(128, 128, 0, 0);  // S, dP
    constexpr uint32_t id_kmn = make_idesc_bf16(128, 64, 0, 1);  // dQ
    constexpr uint32_t id_mnmn = make_idesc_bf16(128, 64, 1, 1); // dV, dK
    mbar_wait(ld_a, 0);
    tc_fence_after();
    // descriptor bases; the start-address field counts 16-byte units (a 16 KB tile = 1024, 2 KB = 128, 32 B = 2)
    const uint64_t kQ = make_smem_desc_sw128(smem_u32(sQ), 16, 1024), kK = make_smem_desc_sw128(smem_u32(sK), 16, 1024);
    const uint64_t kV = make_smem_desc_sw128(smem_u32(sV), 16, 1024), kG = make_smem_desc_sw128(smem_u32(sG), 16, 1024);
    const uint64_t kDs = make_smem_desc_sw128(smem_u32(sDs), 16, 1024);
    const uint64_t mQ = make_smem_desc_sw128(smem_u32(sQ), 8192, 1024), mK = make_smem_desc_sw128(smem_u32(sK), 8192, 1024);
    const uint64_t mG = make_smem_desc_sw128(smem_u32(sG), 8192, 1024);
    const uint64_t mPd = make_smem_desc_sw128(smem_u32(sPd), 16384, 1024), mDs = make_smem_desc_sw128(smem_u32(sDs), 16384, 1024);
    // S = Q_i K_j^T and dP = dO_i V_j^T: rows = queries, so the softmax statistics, the causal test and the dropout
    // groups (which run along the key axis) are per-thread like in forward
    auto issue_s_dp = [&](int pr) {
      const int i = pr == 0 ? 0 : 1, j = pr == 2 ? 1 : 0;
      if (elect_one()) {
#pragma unroll
        for (int k = 0; k < 4; ++k)
          tc_mma_bf16(tmem + TM_ST, kQ + (uint64_t)(i * 1024 + k * 2), kK + (uint64_t)(j * 1024 + k * 2), id_kk, k > 0);
#pragma unroll
        for (int k = 0; k < 4; ++k)
          tc_mma_bf16(tmem + TM_DP, kG + (uint64_t)(i * 1024 + k * 2), kV + (uint64_t)(j * 1024 + k * 2), id_kk, k > 0);
        tc_commit(st_full);
      }
      __syncwarp();
    };
    issue_s_dp(0);
    for (int pr = 0; pr < npair; ++pr) {
      const int i = pr == 0 ? 0 : 1, j = pr == 2 ? 1 : 0;
      mbar_wait(ps_full, pr & 1);  // Pd / dS of this pair are in shared memory; S / dP have been consumed
      // S / dP of the NEXT pair go first: the compute threads turn them into Pd / dS while the accumulate MMAs
      // below still run (they hold their results in registers until acc_free says the tiles may be rewritten)
      if (pr + 1 < npair) {
        mbar_wait(pr + 1 == 1 ? ld_b : ld_c, 0);
        tc_fence_after();
        issue_s_dp(pr + 1);
      }
      if (pr > 0) mbar_wait(drained, (pr - 1) & 1);
      tc_fence_after();
      const uint32_t acc_vk = (pr == 1) ? 1u : 0u;  // second pair of key tile 0 accumulates
      const uint32_t acc_q = (pr == 2) ? 1u : 0u;   // second pair of query tile 1 accumulates
      if (elect_one()) {
        // dV_j += Pd^T dO_i, dK_j += dS^T Q_i: A = the [q x kv] tile read MN-major (M = kv: 64-wide
        // chunks 16 KB apart, K = q rows); B = dO_i / Q_i read MN-major (N = d, K = q rows)
#pragma unroll
        for (int k = 0; k < 8; ++k)
          tc_mma_bf16(tmem + TM_DV, mPd + (uint64_t)(k * 128), mG + (uint64_t)(i * 1024 + k * 128), id_mnmn, acc_vk | (k > 0));
#pragma unroll
        for (int k = 0; k < 8; ++k)
          tc_mma_bf16(tmem + TM_DK, mDs + (uint64_t)(k * 128), mQ + (uint64_t)(i * 1024 + k * 128), id_mnmn, acc_vk | (k > 0));
        // dQ_i += dS K_j: A = dS K-major over kv (two 64-wide k-blocks), B = K_j MN-major (N = d, K = kv rows)
#pragma unroll
        for (int k = 0; k < 8; ++k)
          tc_mma_bf16(tmem + TM_DQ, kDs + (uint64_t)((k >> 2) * 1024 + (k & 3) * 2), mK + (uint64_t)(j * 1024 + k * 128), id_kmn,
                      acc_q | (k > 0));
        tc_commit(acc_free);
        if (pr == npair - 1) tc_commit(acc_done);
      }
      __syncwarp();
    }
  } else {
    // ------------------------------ 256 compute threads --------------------------------
    const int cw = warp - 2;            // 0..7
    const int quad = warp & 3;          // TMEM lane quadrant of this warp
    const int half = cw >> 2;           // which 64 of the 128 key columns (and of the 64 head dims when draining)
    const int rowl = quad * 32 + lane;  // accumulator row inside the tile (query row for S/dP/dQ, key row for dV/dK)
    const int ct = threadIdx.x - 64;    // 0..255
    const uint32_t lane_addr = tmem + ((uint32_t)(quad * 32) << 16);
    uint64_t seed = p.seed;
    if (DROP && p.seed_dev) seed += *p.seed_dev;
    // log-sum-exp of every query row, fetched while the tiles are still in flight (one row per thread)
    if (ct < p.T) lse_s[ct] = p.lse[((int64_t)b * p.NH + h) * p.T + ct] * kLog2e;
    // D_i = dO_i . O_i for every query row of tile tl, read back from the TMA-loaded (swizzled) tiles
    auto compute_D = [&](int tl, const uint8_t* o_tile) {
      if (ct < QT) {
        const int r = ct;
        const uint8_t* gr = sG + tl * 16384 + r * 128;
        const uint8_t* orow = o_tile + r * 128;
        float acc = 0.f;
#pragma unroll
        for (int c = 0; c < 8; ++c) {
          const int off = (c ^ (r & 7)) << 4;
          const uint4 g = *reinterpret_cast<const uint4*>(gr + off), o = *reinterpret_cast<const uint4*>(orow + off);
          const uint32_t gw[4] = {g.x, g.y, g.z, g.w}, ow[4] = {o.x, o.y, o.z, o.w};
#pragma unroll
          for (int t = 0; t < 4; ++t) {
            const float2 gf = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&gw[t]));
            const float2 of = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&ow[t]));
            acc = fmaf(gf.x, of.x, acc);
            acc = fmaf(gf.y, of.y, acc);
          }
        }
        D_s[tl * QT + r] = acc;
      }
      asm volatile("bar.sync 1, 256;" ::: "memory");  // D/lse visible; the O tile may now be overwritten
    };
    BTS(1);
    mbar_wait(ld_a, 0);
    BTS(2);
    compute_D(0, sPd);
    const float sc = p.scale * kLog2e;
    int n_stores = 0;

    // 128 x 64 fp32 accumulator -> bf16 -> swizzled staging tile -> one TMA store
    auto drain = [&](uint32_t tm_col, const CUtensorMap* map, int tile) {
      uint32_t r[32];
      tmem_ld32(lane_addr + tm_col + half * 32, r);
      if (n_stores > 0) {  // the previous store must have finished reading the staging tile
        if (ct == 0) bulk_wait_read<0>();
        asm volatile("bar.sync 1, 256;" ::: "memory");
      }
      tmem_ld_wait();
      uint8_t* rp = sSt + rowl * 128;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        uint4 w;
        w.x = pack_bf16(__uint_as_float(r[8 * j]), __uint_as_float(r[8 * j + 1]));
        w.y = pack_bf16(__uint_as_float(r[8 * j + 2]), __uint_as_float(r[8 * j + 3]));
        w.z = pack_bf16(__uint_as_float(r[8 * j + 4]), __uint_as_float(r[8 * j + 5]));
        w.w = pack_bf16(__uint_as_float(r[8 * j + 6]), __uint_as_float(r[8 * j + 7]));
        *reinterpret_cast<uint4*>(rp + (((half * 4 + j) ^ (rowl & 7)) << 4)) = w;
      }
      fence_proxy_async();
      asm volatile("bar.sync 1, 256;" ::: "memory");
      if (ct == 0) {
        tma_store_2d(map, sSt, h * HD, row0 + tile * QT);
        bulk_commit();
      }
      ++n_stores;
    };

    BTS(3);
    for (int pr = 0; pr < npair; ++pr) {
      const int i = pr == 0 ? 0 : 1, j = pr == 2 ? 1 : 0;
      if (pr == 1) {               // D of query tile 1 (its O tile sits in the staging tile until the first drain)
        mbar_wait(ld_b, 0);
        compute_D(1, sSt);
      }
      BTS(4 + 4 * pr);
      mbar_wait(st_full, pr & 1);
      BTS(5 + 4 * pr);
      tc_fence_after();
      const int qi = i * QT + rowl;  // this thread's query row
      const float lse2 = lse_s[qi], Dq = D_s[qi];
      const uint64_t base = (((uint64_t)b * p.NH + h) * p.T + qi) * (uint64_t)p.T + (uint64_t)(j * QT);
      float pd[32], ds[32];
      // first chunk: math into registers -- the accumulate MMAs of the previous pair may still be reading Pd / dS
      if (i == j) bwd_chunk_math<true, DROP>(p, lane_addr + TM_ST, lane_addr + TM_DP, rowl, half * 64, sc, lse2, Dq, seed, base, pd, ds);
      else bwd_chunk_math<false, DROP>(p, lane_addr + TM_ST, lane_addr + TM_DP, rowl, half * 64, sc, lse2, Dq, seed, base, pd, ds);
      if (pr > 0) {
        mbar_wait(acc_free, (pr - 1) & 1);  // previous pair's accumulators final, its Pd / dS tiles free
        tc_fence_after();
        if (pr == 1) {             // (0,0) finished query tile 0
          drain(TM_DQ, &map_dq, 0);
        } else {                   // (1,0) finished key tile 0
          drain(TM_DV, &map_dv, 0);
          drain(TM_DK, &map_dk, 0);
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(drained);
      }
      BTS(6 + 4 * pr);
      store_row32_sw128(sPd, rowl, half * 64, pd);
      store_row32_sw128(sDs, rowl, half * 64, ds);
      if (i == j) bwd_chunk_math<true, DROP>(p, lane_addr + TM_ST, lane_addr + TM_DP, rowl, half * 64 + 32, sc, lse2, Dq, seed, base, pd, ds);
      else bwd_chunk_math<false, DROP>(p, lane_addr + TM_ST, lane_addr + TM_DP, rowl, half * 64 + 32, sc, lse2, Dq, seed, base, pd, ds);
      store_row32_sw128(sPd, rowl, half * 64 + 32, pd);
      store_row32_sw128(sDs, rowl, half * 64 + 32, ds);
      fence_proxy_async();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(ps_full);
      BTS(7 + 4 * pr);
    }
    BTS(16);
    mbar_wait(acc_done, 0);
    BTS(17);
    tc_fence_after();
    const int last = ntile - 1;
    {
      // the last three accumulators leave together: dV -> the Pd tile, dK -> the dS tile (no MMA reads them any
      // more), dQ -> the staging tile; one fence and one barrier, then three TMA stores
      if (n_stores > 0) {
        if (ct == 0) bulk_wait_read<0>();
        asm volatile("bar.sync 1, 256;" ::: "memory");
      }
      uint8_t* tiles[3] = {sPd, sDs, sSt};
      const uint32_t cols[3] = {TM_DV, TM_DK, TM_DQ};
#pragma unroll
      for (int q = 0; q < 3; ++q) {
        uint32_t r[32];
        tmem_ld32(lane_addr + cols[q] + half * 32, r);
        tmem_ld_wait();
        uint8_t* rp = tiles[q] + rowl * 128;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          uint4 w;
          w.x = pack_bf16(__uint_as_float(r[8 * j]), __uint_as_float(r[8 * j + 1]));
          w.y = pack_bf16(__uint_as_float(r[8 * j + 2]), __uint_as_float(r[8 * j + 3]));
          w.z = pack_bf16(__uint_as_float(r[8 * j + 4]), __uint_as_float(r[8 * j + 5]));
          w.w = pack_bf16(__uint_as_float(r[8 * j + 6]), __uint_as_float(r[8 * j + 7]));
          *reinterpret_cast<uint4*>(rp + (((half * 4 + j) ^ (rowl & 7)) << 4)) = w;
        }
      }
      fence_proxy_async();
      asm volatile("bar.sync 1, 256;" ::: "memory");
      if (ct == 0) {
        tma_store_2d(&map_dv, sPd, h * HD, row0 + last * QT);
        tma_store_2d(&map_dk, sDs, h * HD, row0 + last * QT);
        tma_store_2d(&map_dq, sSt, h * HD, row0 + last * QT);
        bulk_commit();
      }
    }
    if (ct == 0) bulk_wait<0>();
    BTS(18);
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc<512>(tmem);
  }
}

// ===========================================================================
// host
// ===========================================================================
bool attn_tc_supported(const dgpt_attn_args* a) {
  if (a->dtype != DGPT_BF16 || a->H != HD || a->Tq != a->Tk) return false;
  if (a->Tk != 128 && a->Tk != 256) return false;
  const int64_t T = a->Tk;
  auto ok = [&](const void* ptr, int64_t bs, int64_t rs) {
    return ptr && ((uintptr_t)ptr & 15) == 0 && rs % 8 == 0 && bs == T * rs;
  };
  if (!ok(a->q, a->q_bs, a->q_rs) || !ok(a->k, a->k_bs, a->k_rs) || !ok(a->v, a->v_bs, a->v_rs) ||
      !ok(a->o, a->o_bs, a->o_rs))
    return false;
  if (a->d_o) {  // backward call
    if (!ok(a->d_o, a->do_bs, a->do_rs) || !ok(a->dq, a->dq_bs, a->dq_rs) || !ok(a->dk, a->dk_bs, a->dk_rs) ||
        !ok(a->dv, a->dv_bs, a->dv_rs) || !a->lse)
      return false;
  }
  return true;
}

static AttnTcP make_tc_params(const dgpt_attn_args* a) {
  AttnTcP p;
  p.o = a->o; p.dq = a->dq; p.dk = a->dk; p.dv = a->dv; p.o_in = a->o; p.d_o = a->d_o; p.lse = a->lse;
  p.o_rs = a->o_rs; p.dq_rs = a->dq_rs; p.dk_rs = a->dk_rs; p.dv_rs = a->dv_rs; p.do_rs = a->do_rs;
  p.B = a->B; p.NH = a->NH; p.T = a->Tk;
  p.scale = a->scale; p.inv_keep = 1.f / (1.f - a->dropout_p);
  p.thr = dropout_threshold(a->dropout_p); p.site = a->site; p.seed = a->seed; p.seed_dev = a->seed_dev;
  return p;
}

int launch_attn_fwd_tc(const dgpt_attn_args* a, cudaStream_t st) {
  CUtensorMap mq, mk, mv;
  const int64_t rows = (int64_t)a->B * a->Tk, cols = (int64_t)a->NH * HD;
  int rc;
  if ((rc = make_tmap_bf16_2d(&mq, a->q, cols, rows, a->q_rs, 32))) return rc;  // 32-row blocks (see the producer)
  if ((rc = make_tmap_bf16_2d(&mk, a->k, cols, rows, a->k_rs, QT))) return rc;
  if ((rc = make_tmap_bf16_2d(&mv, a->v, cols, rows, a->v_rs, 64))) return rc;
  AttnTcP p = make_tc_params(a);
  static bool attr = false;
  if (!attr) {
    cudaError_t e = cudaFuncSetAttribute(attn_fwd_tc2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kFwd2Smem);
    if (e != cudaSuccess) { set_error("attn_fwd_tc2: smem attribute: %s", cudaGetErrorString(e)); return DGPT_E_LAUNCH; }
    attr = true;
  }
  const int ntile = a->Tk / QT, bh = a->B * a->NH;
  FwdSched sc;
  sc.nheavy = ntile > 1 ? bh : 0;
  sc.nlight = bh;
  sc.probe = clock_probe_buffer();
  int sms = dgpt_sm_count();
  if (sms <= 0) sms = 148;
  const int grid = min(sms, sc.nheavy + sc.nlight);
  launch_pdl(attn_fwd_tc2_kernel, dim3(grid), dim3(kFwd2Threads), kFwd2Smem, st, mq, mk, mv, p, sc);
  return check_launch("attn_fwd_tc2");
}

int launch_attn_bwd_tc(const dgpt_attn_args* a, cudaStream_t st) {
  CUtensorMap mq, mk, mv, mg, mo, mdq, mdk, mdv;
  const int64_t rows = (int64_t)a->B * a->Tk, cols = (int64_t)a->NH * HD;
  int rc;
  if ((rc = make_tmap_bf16_2d(&mq, a->q, cols, rows, a->q_rs, QT))) return rc;
  if ((rc = make_tmap_bf16_2d(&mk, a->k, cols, rows, a->k_rs, QT))) return rc;
  if ((rc = make_tmap_bf16_2d(&mv, a->v, cols, rows, a->v_rs, QT))) return rc;
  if ((rc = make_tmap_bf16_2d(&mg, a->d_o, cols, rows, a->do_rs, QT))) return rc;
  if ((rc = make_tmap_bf16_2d(&mo, a->o, cols, rows, a->o_rs, QT))) return rc;
  if ((rc = make_tmap_bf16_2d(&mdq, a->dq, cols, rows, a->dq_rs, QT))) return rc;
  if ((rc = make_tmap_bf16_2d(&mdk, a->dk, cols, rows, a->dk_rs, QT))) return rc;
  if ((rc = make_tmap_bf16_2d(&mdv, a->dv, cols, rows, a->dv_rs, QT))) return rc;
  static bool attr = false;
  if (!attr) {
    cudaError_t e = cudaFuncSetAttribute(attn_bwd_tc_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kBwdSmem);
    if (e == cudaSuccess)
      e = cudaFuncSetAttribute(attn_bwd_tc_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kBwdSmem);
    if (e != cudaSuccess) { set_error("attn_bwd_tc: smem attribute: %s", cudaGetErrorString(e)); return DGPT_E_LAUNCH; }
    attr = true;
  }
  AttnTcP p = make_tc_params(a);
  dim3 grid(a->NH, a->B);
  if (p.thr) launch_pdl(attn_bwd_tc_kernel<true>, grid, dim3(kBwdThreads), kBwdSmem, st, mq, mk, mv, mg, mo, mdq, mdk, mdv, p);
  else launch_pdl(attn_bwd_tc_kernel<false>, grid, dim3(kBwdThreads), kBwdSmem, st, mq, mk, mv, mg, mo, mdq, mdk, mdv, p);
#ifdef DGPT_ATTN_TS
  {
    cudaStreamSynchronize(st);
    long long h[64];
    cudaMemcpyFromSymbol(h, g_attn_ts, sizeof(h));
    printf("attn bwd CTA: setup %lld | load wait %lld | D %lld |", h[1] - h[0], h[2] - h[1], h[3] - h[2]);
    for (int pr = 0; pr < 3; ++pr)
      printf(" pair%d: S/dP wait %lld, drains %lld, chunks %lld |", pr, h[5 + 4 * pr] - h[4 + 4 * pr], h[6 + 4 * pr] - h[5 + 4 * pr],
             h[7 + 4 * pr] - h[6 + 4 * pr]);
    printf(" acc wait %lld | final drains %lld | total %lld\n", h[17] - h[16], h[18] - h[17], h[18] - h[0]);
    fflush(stdout);
  }
#endif
  return check_launch("attn_bwd_tc");
}

}  // namespace dgpt
