// Tensor-mode GEMM for sm_100a: bf16 operands staged by TMA (128B swizzle) into a
// multi-stage shared-memory ring, tcgen05.mma (cta_group::1, 128 x BN x 16) issued
// by one thread with fp32 accumulators in TMEM, and a fused epilogue
// (bias / ReLU / ReLU-mask / dropout / residual) whose results leave the SM through
// swizzled shared-memory staging tiles and TMA stores -- or TMA fp32 reduce-adds for
// split-K / accumulate -- so the output is written in full 128-byte lines, clipped at the
// matrix edge by the tensor map, with no per-thread global stores.  Persistent: one CTA
// per SM walks the tile list; TMEM holds two accumulators so the epilogue of tile i
// overlaps the mainloop of tile i+1.  Long-K GEMMs of the big activations use 256-row
// CTA tiles (two M = 128 MMAs per k-step on one B stage, see TcCfg), and wgrads can
// carry the bias gradient as a column-sum MMA.
//
// Warp roles (320 threads): warp 0 = TMA producer, warp 1 = TMEM owner + MMA
// issuer, warps 2..9 = epilogue (TMEM lane quadrant = warp_id % 4, two warps per quadrant).
//
// Operand layouts: K-major ([rows, K], K contiguous: activations, nn.Linear
// weights) and MN-major ([K, rows], rows contiguous: the transposed views that
// dgrad / wgrad need) are both fed straight from the row-major tensors -- no
// transposed copies are ever written to HBM.
#include <cuda.h>

#include "epilogue.cuh"
#include "ptx.cuh"

namespace dgpt {

using namespace ptx;

static constexpr int TBM = 128;       // tile M (UMMA M)
static constexpr int TBK = 64;        // k-block: 64 bf16 = one 128-byte swizzle row
static constexpr int UMMA_K = 16;
static constexpr int kThreads = 64 + 256;  // TMA warp, MMA warp, 8 epilogue warps
static constexpr int kSmemMax = 232448;    // 227 KB per CTA on sm_100

enum StoreMode { kStoreDirect = 0, kStoreTma = 1, kStoreTmaAdd = 2 };

struct TcParams {
  int M, N, K;
  int m_tiles, n_tiles, split_k, kb_total, kb_per_split;
  int vec_ok;      // epilogue operands (bias / residual) allow the vector fast path
  int store_mode;  // StoreMode for D
  unsigned long long* probe; // DGPT_CLOCK_PROBE stamps (or NULL)
  uint32_t* mask_out;        // ReLU bit mask written by the forward GEMM  [(n / 32) * M + m]
  const uint32_t* mask_in;   // ... and applied by the dgrad GEMM
  float* a_colsum;           // out[m] += sum_k A[m, k]  (bias gradient riding on the wgrad GEMM, CS instantiations)
  Epilogue ep;
};

// epilogue feature bits (compile-time mask of the fused epilogue, or -1 = generic element-wise path)
enum { kEpiBias = 1, kEpiRelu = 2, kEpiAux = 4, kEpiDrop = 8, kEpiRes = 16, kEpiMaskIn = 32, kEpiMaskOut = 64 };

// EPI: epilogue feature mask (see the kernel).  With kEpiRes the fp32 residual operand arrives by TMA into the
// epilogue staging buffers, see the epilogue below: the next tile's residual is fetched once this tile's stores have
// been read out of them.
// TM = 128-row sub-tiles per CTA tile (1 or 2).  TM = 2: a 256 x BN tile as two M = 128 MMAs per k-step that share one
// B stage -- 2/3 of the operand bytes per MMA cycle of a 128 x BN tile (measured: the mainloop of 128-row tiles waits
// for operands 30-50 % of the time, the SM ingests ~70 B/cycle and a 128 x 256 tile needs 94).  The two accumulators
// fill TMEM (2 x 256 or 2 x 192 columns), so TM = 2 tiles are single-buffered: the epilogue of a tile does not overlap
// the mainloop of the next one, which costs little because such GEMMs are launched with <= ~3 tiles per CTA.
template <int BN, int EPI, int CS = 0, int TM = 1>
struct TcCfg {
  static constexpr bool kRes = EPI >= 0 && (EPI & kEpiRes) != 0;
  static constexpr int kABytes = TM * TBM * TBK * 2;
  static constexpr int kBBytes = BN * TBK * 2;
  static constexpr int kStageBytes = kABytes + kBBytes;
  // 4 KB staging buffers per epilogue warp: 2, or (residual epilogues) one per fp32 block of the warp's half of a
  // tile; TM = 2 keeps one (the ring needs the room)
  static constexpr int kResBlocks = BN / 2 / 32;
  static constexpr int kStagingBufs = kRes ? kResBlocks : (TM == 2 ? 1 : 2);
  static constexpr int kStagingBytes = 8 * kStagingBufs * 4096;
  static constexpr int kBiasBytes = 2 * BN * 4;  // bias slice of the tile, double-buffered with the accumulator
  static constexpr int kBarBytes = 512;
  static constexpr int kRing = kSmemMax - kStagingBytes - kBiasBytes - kBarBytes;
  static constexpr int kStages = kRing / kStageBytes > 8 ? 8 : kRing / kStageBytes;
  // accumulator buffers: two when they fit the 512 TMEM columns (+ 16 column-sum columns per sub-tile and buffer with CS)
  static constexpr int kNAcc = (2 * TM * BN + (CS ? 2 * TM * 16 : 0) <= 512) ? 2 : 1;
  static constexpr int kTmemNeed = kNAcc * TM * BN + (CS ? kNAcc * TM * 16 : 0);
  static constexpr int kTmemCols = kTmemNeed <= 32 ? 32 : kTmemNeed <= 64 ? 64 : kTmemNeed <= 128 ? 128 : kTmemNeed <= 256 ? 256 : 512;
  static_assert(kTmemNeed <= 512, "no TMEM room");
  static_assert(TM == 1 || !kRes, "256-row CTA tiles: no TMA-fed residual");
  static constexpr size_t kSmemBytes = (size_t)kStages * kStageBytes + kStagingBytes + kBiasBytes + kBarBytes;
  static_assert(kStages >= 3, "shared-memory ring too shallow");
};

// --------------------------------------------------------------------------
// Fast epilogue math on 32 consecutive accumulator columns [n, n+32) of row m, in registers.
// Order (= epilogue_value): + bias, ReLU (+ bit mask out), bit mask in, dropout, + residual.
//   bias_s  : the tile's bias slice in shared memory (broadcast reads)
//   res_row : this row of the 32 x 32 fp32 residual block the TMA put into the staging buffer (SW128)
// Keep this small: the kernel's instruction footprint must stay inside the instruction cache.
// --------------------------------------------------------------------------
template <int EPI>
__device__ __forceinline__ void epi_math32(const Epilogue& e, int m, int n, uint32_t (&r)[32], const float* bias_s,
                                           const uint8_t* res_row, int row7, uint32_t mask_in, uint32_t& mask_out) {
  if (EPI & kEpiBias) {
#pragma unroll
    for (int j = 0; j < 32; j += 4) {
      const float4 b = *reinterpret_cast<const float4*>(bias_s + j);  // shared-memory broadcast
      r[j] = __float_as_uint(__uint_as_float(r[j]) + b.x);
      r[j + 1] = __float_as_uint(__uint_as_float(r[j + 1]) + b.y);
      r[j + 2] = __float_as_uint(__uint_as_float(r[j + 2]) + b.z);
      r[j + 3] = __float_as_uint(__uint_as_float(r[j + 3]) + b.w);
    }
  }
  if (EPI & kEpiMaskOut) {
    uint32_t mk = 0;
#pragma unroll
    for (int j = 0; j < 32; ++j) mk |= (__uint_as_float(r[j]) > 0.f) ? (1u << j) : 0u;
    mask_out = mk;
  }
  if (EPI & kEpiRelu) {
#pragma unroll
    for (int j = 0; j < 32; ++j) r[j] = __float_as_uint(fmaxf(__uint_as_float(r[j]), 0.f));
  }
  if (EPI & kEpiMaskIn) {
#pragma unroll
    for (int j = 0; j < 32; ++j) r[j] = ((mask_in >> j) & 1u) ? r[j] : 0u;
  }
  if (EPI & kEpiDrop) {
    const uint64_t i0 = (uint64_t)m * (uint64_t)e.N + (uint64_t)n;
    if ((e.N & 31) == 0) {  // the 32 columns are one mask group: one hash, then a multiply-add per element
      const DropGroup g = dropout_group(e.seed, e.site, i0 >> 5);
#pragma unroll
      for (int j = 0; j < 32; ++j)
        r[j] = dropout_word(g, j) >= e.thr ? __float_as_uint(__uint_as_float(r[j]) * e.inv_keep) : 0u;
    } else {
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const u32x4 b = dropout_bits4(e.seed, e.site, (i0 >> 2) + j);
        r[4 * j] = b.x >= e.thr ? __float_as_uint(__uint_as_float(r[4 * j]) * e.inv_keep) : 0u;
        r[4 * j + 1] = b.y >= e.thr ? __float_as_uint(__uint_as_float(r[4 * j + 1]) * e.inv_keep) : 0u;
        r[4 * j + 2] = b.z >= e.thr ? __float_as_uint(__uint_as_float(r[4 * j + 2]) * e.inv_keep) : 0u;
        r[4 * j + 3] = b.w >= e.thr ? __float_as_uint(__uint_as_float(r[4 * j + 3]) * e.inv_keep) : 0u;
      }
    }
  }
  if (EPI & kEpiRes) {
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float4 x = *reinterpret_cast<const float4*>(res_row + ((j ^ row7) << 4));
      r[4 * j] = __float_as_uint(__uint_as_float(r[4 * j]) + x.x);
      r[4 * j + 1] = __float_as_uint(__uint_as_float(r[4 * j + 1]) + x.y);
      r[4 * j + 2] = __float_as_uint(__uint_as_float(r[4 * j + 2]) + x.z);
      r[4 * j + 3] = __float_as_uint(__uint_as_float(r[4 * j + 3]) + x.w);
    }
  }
}

// Ragged edge (n + 32 > N), unaligned operands, outputs the TMA cannot address, the optional second
// output and every combination without its own instantiation: one compact element-wise loop.
// (Epilogue BY VALUE: a reference would pin the caller's copy in local memory.)
__device__ __noinline__ void epilogue_slow32(const Epilogue e, uint32_t* r, int m, int n, int store_main) {
  if (m >= e.M) return;
#pragma unroll 1
  for (int j = 0; j < 32; ++j) {
    if (n + j >= e.N) break;
    const float x = epilogue_value(e, m, n + j, __uint_as_float(r[j]));
    r[j] = __float_as_uint(x);
    if (store_main) {
      const int64_t i = (int64_t)m * e.ldd + n + j;
      if (e.d_dtype == DGPT_F32) {
        float* d = reinterpret_cast<float*>(e.D);
        if (e.atomic) atomicAdd(d + i, x);
        else d[i] = e.accumulate ? d[i] + x : x;
      } else {
        reinterpret_cast<__nv_bfloat16*>(e.D)[i] = __float2bfloat16_rn(x);
      }
    }
    if (e.D2) {
      const int64_t i = (int64_t)m * e.ldd2 + n + j;
      if (e.d2_dtype == DGPT_F32) reinterpret_cast<float*>(e.D2)[i] = x;
      else reinterpret_cast<__nv_bfloat16*>(e.D2)[i] = __float2bfloat16_rn(x);
    }
  }
}

__device__ __forceinline__ uint32_t pack2(uint32_t a, uint32_t b) {
  __nv_bfloat162 t = __floats2bfloat162_rn(__uint_as_float(a), __uint_as_float(b));
  return *reinterpret_cast<uint32_t*>(&t);
}

// one row (128 bytes) of a 32-row SWIZZLE_128B staging tile
__device__ __forceinline__ void stage_row_f32(uint8_t* tile, int row, const uint32_t (&v)[32]) {
  uint8_t* rp = tile + row * 128;
#pragma unroll
  for (int j = 0; j < 8; ++j)
    *reinterpret_cast<uint4*>(rp + ((j ^ (row & 7)) << 4)) = make_uint4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
}
__device__ __forceinline__ void stage_half_row_bf16(uint8_t* tile, int row, int half, const uint32_t (&v)[32]) {
  uint8_t* rp = tile + row * 128;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    uint4 w;
    w.x = pack2(v[8 * j], v[8 * j + 1]); w.y = pack2(v[8 * j + 2], v[8 * j + 3]);
    w.z = pack2(v[8 * j + 4], v[8 * j + 5]); w.w = pack2(v[8 * j + 6], v[8 * j + 7]);
    *reinterpret_cast<uint4*>(rp + (((half * 4 + j) ^ (row & 7)) << 4)) = w;
  }
}

// every split owns at least one k-block (launch_gemm_tc re-derives split_k from kb_per_split)
__device__ __forceinline__ bool kb_nonempty(const TcParams& p, int ks) { return ks * p.kb_per_split < p.kb_total; }

// --------------------------------------------------------------------------
// the kernel
//   EPI  : compile-time epilogue feature mask (fast path), or -1 = generic element-wise epilogue
//   OBF  : output element type of the fast path (1 = bf16, 0 = fp32); ignored when EPI < 0
//   CS   : 1 = column sums, see below
//   TM   : 128-row sub-tiles per CTA tile (see TcCfg)
// --------------------------------------------------------------------------
// CS = 1 (wgrad form: A MN-major, plain fp32 epilogue): the column sums of the stored A matrix
// (= row sums of the logical A: sum_k A[m, k], the bias gradient when A = dY^T) ride on the tensor core as
// one extra N = 16 MMA per k-step against an all-ones B tile -- no separate pass over dY.
template <int BN, int A_MN, int B_MN, int EPI, int OBF, int CS, int TM>
__global__ void __launch_bounds__(kThreads, 1)
gemm_tc_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b,
               const __grid_constant__ CUtensorMap map_d, const __grid_constant__ CUtensorMap map_r, TcParams p) {
  using Cfg = TcCfg<BN, EPI, CS, TM>;
  constexpr bool kRes = Cfg::kRes;
  static_assert(!CS || EPI == 0, "column sums: plain epilogue");
  constexpr int kStages = Cfg::kStages;
  constexpr int kABytes = Cfg::kABytes;
  constexpr int kNAcc = Cfg::kNAcc;
  constexpr int kTileM = TBM * TM;        // rows of a CTA tile
  constexpr int kAccCols = TM * BN;       // TMEM columns of one accumulator buffer
  constexpr int kBBytes = Cfg::kBBytes;
  constexpr uint32_t kIdesc = make_idesc_bf16(TBM, BN, A_MN, B_MN);

  extern __shared__ __align__(1024) uint8_t smem[];  // SWIZZLE_128B tiles need 1024-byte alignment
  uint8_t* stage_base = smem;
  uint8_t* staging = smem + (size_t)kStages * Cfg::kStageBytes;  // 1024-aligned: stage sizes are multiples of 8 KB
  float* bias_s = reinterpret_cast<float*>(staging + Cfg::kStagingBytes);  // [2][BN]
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(staging + Cfg::kStagingBytes + Cfg::kBiasBytes);
  uint64_t* empty_bar = full_bar + 8;
  uint64_t* tmem_full = empty_bar + 8;
  uint64_t* tmem_empty = tmem_full + 2;
  uint64_t* res_bar = tmem_empty + 2;  // [8 epilogue warps]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(res_bar + 8);

  clock_probe_begin(p.probe);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (threadIdx.x == 0) {
    prefetch_tensormap(&map_a);
    prefetch_tensormap(&map_b);
    if (p.store_mode != kStoreDirect) prefetch_tensormap(&map_d);
    if (kRes) prefetch_tensormap(&map_r);
    for (int s = 0; s < kStages; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&tmem_full[i], 1);
      mbar_init(&tmem_empty[i], 8);  // one arrive per epilogue warp
    }
    for (int i = 0; i < 8; ++i) mbar_init(&res_bar[i], 1);
    fence_barrier_init();
  }
  if (CS && warp >= 2) {
    // all-ones bf16 tile (8 rows x 128 B, every layout of it is the same tile) in the unused bias region
    uint32_t* ones = reinterpret_cast<uint32_t*>(bias_s);
    for (int i = (warp - 2) * 32 + lane; i < 256; i += 256) ones[i] = 0x3F803F80u;
    fence_proxy_async();  // generic-proxy writes -> visible to the MMA's async-proxy reads (after the barrier below)
  }
  if (warp == 1) tmem_alloc<Cfg::kTmemCols>(tmem_slot);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  // everything above touched only this CTA's shared memory / TMEM: with programmatic dependent launch it overlapped
  // the tail of the previous kernel in the stream; from here on global memory is read and written
  pdl_launch_dependents();
  pdl_wait();

  const bool prof = p.probe != nullptr && blockIdx.x == 0;  // DGPT_CLOCK_PROBE: where the roles of CTA 0 wait
  const int tiles_mn = p.m_tiles * p.n_tiles;
  const int total_tiles = tiles_mn * p.split_k;
  const int t_first = blockIdx.x, t_step = gridDim.x;

  if (warp == 0) {
    // ------------------------------ TMA producer ---------------------------
    // the whole warp walks the loop (uniform control flow); one elected lane issues
    int s = 0;
    uint32_t ph = 0;
    long long pr_wait = 0;
    const long long pr_t0 = prof ? clock64() : 0;
    for (int t = t_first; t < total_tiles; t += t_step) {
      const int ks = t / tiles_mn, mn = t - ks * tiles_mn;
      const int m0 = (mn / p.n_tiles) * kTileM, n0 = (mn % p.n_tiles) * BN;
      const int kb0 = ks * p.kb_per_split, kb1 = min(p.kb_total, kb0 + p.kb_per_split);
      for (int kb = kb0; kb < kb1; ++kb) {
        const long long tw0 = prof ? clock64() : 0;
        mbar_wait(&empty_bar[s], ph ^ 1);
        if (prof) pr_wait += clock64() - tw0;
        uint8_t* sa = stage_base + (size_t)s * Cfg::kStageBytes;
        uint8_t* sb = sa + kABytes;
        const int k0 = kb * TBK;
        if (elect_one()) {
          mbar_expect_tx(&full_bar[s], kABytes + kBBytes);
          if (A_MN) {
#pragma unroll
            for (int c = 0; c < kTileM / 64; ++c) tma_load_2d(sa + c * 8192, &map_a, &full_bar[s], m0 + c * 64, k0);
          } else {
#pragma unroll
            for (int mi = 0; mi < TM; ++mi) tma_load_2d(sa + mi * 16384, &map_a, &full_bar[s], k0, m0 + mi * TBM);
          }
          if (B_MN) {
#pragma unroll
            for (int c = 0; c < BN / 64; ++c) tma_load_2d(sb + c * 8192, &map_b, &full_bar[s], n0 + c * 64, k0);
          } else {
            tma_load_2d(sb, &map_b, &full_bar[s], k0, n0);
          }
        }
        __syncwarp();
        if (++s == kStages) { s = 0; ph ^= 1; }
      }
    }
    if (prof && lane == 0) { p.probe[24] = (unsigned long long)(clock64() - pr_t0); p.probe[25] = (unsigned long long)pr_wait; }
  } else if (warp == 1) {
    // ------------------------------ MMA issuer -----------------------------
    // the whole warp walks the loop; one elected lane issues
    int s = 0;
    uint32_t ph = 0;
    int acc = 0;
    uint32_t acc_ph = 0;
    long long mm_wacc = 0, mm_wfull = 0;
    const long long mm_t0 = prof ? clock64() : 0;
    for (int t = t_first; t < total_tiles; t += t_step) {
      const int ks = t / tiles_mn;
      const int kb0 = ks * p.kb_per_split, kb1 = min(p.kb_total, kb0 + p.kb_per_split);
      const bool cs_tile = CS && ((t - ks * tiles_mn) % p.n_tiles) == 0;  // column sums: once per row tile
      const long long ta0 = prof ? clock64() : 0;
      mbar_wait(&tmem_empty[acc], acc_ph ^ 1);
      if (prof) mm_wacc += clock64() - ta0;
      tc_fence_after();
      const uint32_t d_tmem = tmem_base + (uint32_t)(acc * kAccCols);
      for (int kb = kb0; kb < kb1; ++kb) {
        const long long tf0 = prof ? clock64() : 0;
        mbar_wait(&full_bar[s], ph);
        if (prof) mm_wfull += clock64() - tf0;
        tc_fence_after();
        const uint32_t sa = smem_u32(stage_base + (size_t)s * Cfg::kStageBytes);
        const uint32_t sb = sa + kABytes;
        // K-major: 32 bytes per UMMA_K inside the 128B swizzle row, 8-row groups 1024 B apart.
        // MN-major: 16 k-rows (2 KB) per UMMA_K, 64-element MN chunks 8 KB apart.
        // (the start-address field counts 16-byte units: + 2 / + 128 per UMMA_K step)
        const uint64_t da0 = A_MN ? make_smem_desc_sw128(sa, 8192, 1024) : make_smem_desc_sw128(sa, 16, 1024);
        const uint64_t db0 = B_MN ? make_smem_desc_sw128(sb, 8192, 1024) : make_smem_desc_sw128(sb, 16, 1024);
        if (elect_one()) {
#pragma unroll
          for (int k = 0; k < TBK / UMMA_K; ++k) {
            const uint64_t da = da0 + (uint64_t)(k * (A_MN ? 128 : 2));
            const uint64_t db = db0 + (uint64_t)(k * (B_MN ? 128 : 2));
#pragma unroll
            for (int mi = 0; mi < TM; ++mi)  // sub-tile mi: 16 KB (1024 descriptor units) further into the A stage
              tc_mma_bf16(d_tmem + (uint32_t)(mi * BN), da + (uint64_t)(mi * 1024), db, kIdesc, (kb > kb0 || k > 0) ? 1u : 0u);
            if (CS && cs_tile) {
              // ones tile: K-major, N = 16 rows as two aliased 8-row groups (SBO = 0), 32 bytes per UMMA_K
              const uint64_t d1 = make_smem_desc_sw128(smem_u32(bias_s), 16, 0) + (uint64_t)(k * 2);
#pragma unroll
              for (int mi = 0; mi < TM; ++mi)
                tc_mma_bf16(tmem_base + (uint32_t)(kNAcc * kAccCols + (acc * TM + mi) * 16), da + (uint64_t)(mi * 1024), d1,
                            make_idesc_bf16(TBM, 16, A_MN, 0), (kb > kb0 || k > 0) ? 1u : 0u);
            }
          }
          tc_commit(&empty_bar[s]);  // smem stage is free once these MMAs retire
        }
        __syncwarp();
        if (++s == kStages) { s = 0; ph ^= 1; }
      }
      if (elect_one()) tc_commit(&tmem_full[acc]);  // accumulator complete -> epilogue
      __syncwarp();
      if (++acc == kNAcc) { acc = 0; acc_ph ^= 1; }
    }
    if (prof && lane == 0) {
      p.probe[8] = (unsigned long long)(clock64() - mm_t0);
      p.probe[9] = (unsigned long long)mm_wacc;
      p.probe[10] = (unsigned long long)mm_wfull;
    }
  } else {
    // ------------------------------ epilogue -------------------------------
    // Eight warps: TMEM lane quadrant = warp % 4 (hardware rule); the two warps of a quadrant split the tile's
    // columns.  Work unit = one 4 KB staging block: 32 rows x 128 bytes of OUTPUT (64 bf16 / 32 fp32 columns):
    //   tcgen05.ld (TMEM reads are cheap: ~40 cycles for 4 x 32 columns, measured) -> math in registers ->
    //   one swizzled 128-byte row per thread into the block -> fence.proxy.async -> one TMA store / reduce.
    // A warp's blocks rotate through its staging buffers; cp.async.bulk.wait_group.read keeps a buffer from
    // being rewritten while an earlier store still reads it.
    // Residual (kRes): row-strided loads of the fp32 residual cost 32 L1 wavefronts per instruction (measured
    // +18 us on a 9 us GEMM), so the TMA fetches the residual block INTO the staging buffer the output will
    // leave from -- for the NEXT tile, as soon as this tile's stores have been read out -- and the add happens in place.
    const int ew = warp - 2;
    const int quad = warp & 3;   // TMEM lanes [32*quad, 32*quad+32)
    const int half = ew >> 2;    // columns [half*BN/2, (half+1)*BN/2)
    constexpr bool kFast = EPI >= 0;
    // Column split between the two warps of a quadrant.  128- and 256-column tiles: half each.  192-column tiles
    // (the N = 384 GEMMs of this model: 2 tiles per row instead of 3, i.e. A is re-read twice instead of three
    // times and the per-k-block bookkeeping is paid twice instead of three times): 96 fp32 columns each, but bf16
    // output leaves in 64-column blocks, so there the first warp takes 128 columns and the second 64.
    constexpr int kCols = BN == 192 ? 128 : BN / 2;  // upper bound of a warp's columns (array sizes)
    constexpr int CPB = (kFast && OBF) ? 64 : 32;  // accumulator columns per staging block (fast path; residual bookkeeping)
    constexpr int NBLK = (BN / 2) / CPB;            // residual bookkeeping (fp32 output: BN / 2 columns per warp)
    constexpr int kBufs = Cfg::kStagingBufs;
    uint8_t* my_stage = staging + ew * (kBufs * 4096);
    uint64_t* my_res_bar = res_bar + ew;
    int nbuf = 0;
    int acc = 0;
    uint32_t acc_ph = 0;
    int it = 0;
    Epilogue ep = p.ep;
    epilogue_resolve_seed(ep);
    const int mode = p.store_mode;
    const bool out_bf16 = kFast ? (OBF != 0) : (ep.d_dtype == DGPT_BF16);
    const int cpb = out_bf16 ? 64 : 32;  // compile-time on the fast path, run-time in the generic kernel
    const int col_beg = (BN == 192 && out_bf16) ? half * 128 : half * (BN / 2);            // first column of this warp
    const int ncols = (BN == 192 && out_bf16) ? (half ? 64 : 128) : BN / 2;                // ... and how many
    const int nblk = ncols / cpb;
    const int row7 = lane & 7;

    auto res_prefetch = [&](int t) {  // lane 0: residual blocks of tile t -> staging buffers [0, NBLK)
      const int ks = t / tiles_mn, mn = t - ks * tiles_mn;
      const int m0 = (mn / p.n_tiles) * kTileM, n0 = (mn % p.n_tiles) * BN;
      const int nb = n0 + col_beg;
      int cnt = 0;
      for (int b = 0; b < NBLK; ++b) cnt += (nb + b * CPB < p.N) ? 1 : 0;
      if (cnt == 0 || m0 + quad * 32 >= p.M) { mbar_arrive(my_res_bar); return; }
      mbar_expect_tx(my_res_bar, cnt * 4096);
      for (int b = 0; b < NBLK; ++b)
        if (nb + b * CPB < p.N) tma_load_2d(my_stage + b * 4096, &map_r, my_res_bar, nb + b * CPB, m0 + quad * 32);
    };
    if (kRes && lane == 0 && t_first < total_tiles) res_prefetch(t_first);

    long long ep_wfull = 0, ep_wread = 0, ep_wres = 0;
    const long long ep_t0 = prof ? clock64() : 0;
    for (int t = t_first; t < total_tiles; t += t_step, ++it) {
      const int ks = t / tiles_mn, mn = t - ks * tiles_mn;
      const int m0 = (mn / p.n_tiles) * kTileM, n0 = (mn % p.n_tiles) * BN;
      ep.first_split = (ks == 0);
      const int nbeg = n0 + col_beg;
      // stage this tile's bias slice (each warp an eighth) while the accumulator is still being produced
      float* bias_t = bias_s + acc * BN;
      if (kFast && (EPI & kEpiBias)) {
        const int col = ew * (BN / 8) + lane * 4;
        if (lane * 4 < BN / 8 && n0 + col < p.N)  // (BN / 8 = 16, 24 or 32 floats per warp)
          *reinterpret_cast<float4*>(bias_t + col) = __ldg(reinterpret_cast<const float4*>(ep.bias + n0 + col));
        asm volatile("bar.sync 1, 256;" ::: "memory");  // the eight epilogue warps
      }
      uint32_t mk_in_all[TM][kCols / 32];  // (fetched before the accumulator wait: the latency hides behind it)
      if (kFast && (EPI & kEpiMaskIn)) {
#pragma unroll
        for (int mi = 0; mi < TM; ++mi) {
          const int mm = m0 + mi * TBM + quad * 32 + lane;
#pragma unroll
          for (int w = 0; w < kCols / 32; ++w)
            mk_in_all[mi][w] = (mm < p.M && 32 * w < ncols && nbeg + 32 * w < p.N)
                                   ? __ldg(p.mask_in + (size_t)((nbeg >> 5) + w) * p.M + mm) : 0u;
        }
      }
      const long long tr0 = prof ? clock64() : 0;
      if (kRes) mbar_wait(my_res_bar, (uint32_t)it & 1u);
      const long long tr1 = prof ? clock64() : 0;
      mbar_wait(&tmem_full[acc], acc_ph);
      if (prof) { ep_wres += tr1 - tr0; ep_wfull += clock64() - tr1; }
      tc_fence_after();
#pragma unroll
      for (int mi = 0; mi < TM; ++mi) {  // the 128-row sub-tiles of the CTA tile
      const int mrow0 = m0 + mi * TBM + quad * 32;
      const int m = mrow0 + lane;
      const bool active = mrow0 < p.M && nbeg < p.N;
      const uint32_t (&mk_in)[kCols / 32] = mk_in_all[mi];
      const uint32_t row_addr = tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(acc * kAccCols + mi * BN + col_beg);
#pragma unroll 1
      for (int b = 0; b < nblk; ++b) {
        const int n = nbeg + b * cpb;
        const bool in_range = active && n < p.N;
        uint8_t* tile = my_stage + (kRes ? b : nbuf) * 4096;
        if (!in_range) continue;
        uint32_t r0[32], r1[32];
        tmem_ld32(row_addr + b * cpb, r0);
        if (cpb == 64) tmem_ld32(row_addr + b * cpb + 32, r1);
        if (!kRes && mode != kStoreDirect) {
          const long long tb0 = prof ? clock64() : 0;
          if (lane == 0) bulk_wait_read<kBufs - 1>();  // the store that last used this buffer has drained it
          __syncwarp();
          if (prof) ep_wread += clock64() - tb0;
        }
        tmem_ld_wait();
        const bool fast = kFast && p.vec_ok && mode != kStoreDirect && n + cpb <= p.N;
        if (fast) {
          uint32_t mo = 0;
          epi_math32<kFast ? EPI : 0>(ep, m, n, r0, bias_t + col_beg + b * cpb, tile + lane * 128, row7,
                                      (kFast && (EPI & kEpiMaskIn)) ? mk_in[(b * cpb) >> 5] : 0u, mo);
          if (kFast && (EPI & kEpiMaskOut)) {
            if (m < p.M) p.mask_out[(size_t)(n >> 5) * p.M + m] = mo;
          }
          if (cpb == 64) {
            epi_math32<kFast ? EPI : 0>(ep, m, n + 32, r1, bias_t + col_beg + b * cpb + 32, tile + lane * 128, row7,
                                        (kFast && (EPI & kEpiMaskIn)) ? mk_in[((b * cpb) >> 5) + 1] : 0u, mo);
            if (kFast && (EPI & kEpiMaskOut)) {
              if (m < p.M) p.mask_out[(size_t)((n >> 5) + 1) * p.M + m] = mo;
            }
          }
        } else {
          // (through a local copy: passing r0 / r1 themselves would pin them in local memory for the fast path too)
          uint32_t tmp[32];
#pragma unroll
          for (int j = 0; j < 32; ++j) tmp[j] = r0[j];
          epilogue_slow32(ep, tmp, m, n, mode == kStoreDirect);
#pragma unroll
          for (int j = 0; j < 32; ++j) r0[j] = tmp[j];
          if (cpb == 64 && n + 32 < p.N) {
#pragma unroll
            for (int j = 0; j < 32; ++j) tmp[j] = r1[j];
            epilogue_slow32(ep, tmp, m, n + 32, mode == kStoreDirect);
#pragma unroll
            for (int j = 0; j < 32; ++j) r1[j] = tmp[j];
          }
        }
        if (mode == kStoreDirect) continue;
        if (out_bf16) {
          stage_half_row_bf16(tile, lane, 0, r0);
          stage_half_row_bf16(tile, lane, 1, r1);
        } else {
          stage_row_f32(tile, lane, r0);
        }
        fence_proxy_async();
        __syncwarp();
        if (lane == 0) {
          if (mode == kStoreTmaAdd) tma_reduce_add_2d(&map_d, tile, n, mrow0);
          else tma_store_2d(&map_d, tile, n, mrow0);
          bulk_commit();
        }
        if (!kRes) nbuf = (nbuf + 1 == kBufs) ? 0 : nbuf + 1;
      }
      if (CS && n0 == 0 && half == 0 && mrow0 < p.M) {
        const float cs = __uint_as_float(tmem_ld1(tmem_base + ((uint32_t)(quad * 32) << 16) +
                                                  (uint32_t)(kNAcc * kAccCols + (acc * TM + mi) * 16)));
        tmem_ld_wait();
        if (m < p.M && kb_nonempty(p, ks)) atomicAdd(p.a_colsum + m, cs);
      }
      }  // sub-tiles
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        mbar_arrive(&tmem_empty[acc]);
        if (kRes && t + t_step < total_tiles) {
          // residual of the next tile -> the same buffers, once this tile's stores have been read out of them
          bulk_wait_read<0>();
          res_prefetch(t + t_step);
        }
      }
      if (++acc == kNAcc) { acc = 0; acc_ph ^= 1; }
    }
    if (prof && ew == 0 && lane == 0) {
      p.probe[16] = (unsigned long long)(clock64() - ep_t0);
      p.probe[17] = (unsigned long long)ep_wfull;
      p.probe[18] = (unsigned long long)ep_wread;
      p.probe[19] = (unsigned long long)ep_wres;
    }
    const long long td0 = prof ? clock64() : 0;
    if (lane == 0) bulk_wait<0>();  // all output tiles have landed before the CTA retires
    if (prof && ew == 0 && lane == 0) p.probe[20] = (unsigned long long)(clock64() - td0);
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc<Cfg::kTmemCols>(tmem_base);
  }
  clock_probe_end(p.probe);
}

// --------------------------------------------------------------------------
// host side
// --------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode() {
  static EncodeTiledFn fn = nullptr;
  static bool tried = false;
  if (!tried) {
    tried = true;
    void* sym = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &sym, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = (EncodeTiledFn)sym;
    else
      cudaGetLastError();
  }
  return fn;
}

// 2-D tensor map with 128-byte swizzle and zero fill out of bounds: inner (contiguous) extent `inner`
// elements, `outer` rows of pitch ld elements, box = box_inner x box_outer elements (box_inner * esize == 128).
int make_tmap_2d(CUtensorMap* map, const void* base, int dtype, int64_t inner, int64_t outer, int64_t ld,
                 int box_inner, int box_outer) {
  EncodeTiledFn enc = get_encode();
  if (!enc) {
    set_error("cuTensorMapEncodeTiled driver entry point not available");
    return DGPT_E_DEVICE;
  }
  const int esize = dtype == DGPT_F32 ? 4 : 2;
  DGPT_REQUIRE(((uintptr_t)base & 15) == 0 && (ld * esize) % 16 == 0,
               "TMA needs a 16-byte aligned base and row pitch (ld=%lld elements of %d bytes)", (long long)ld, esize);
  cuuint64_t gdim[2] = {(cuuint64_t)inner, (cuuint64_t)outer};
  cuuint64_t gstr[1] = {(cuuint64_t)ld * esize};
  cuuint32_t box[2] = {(cuuint32_t)box_inner, (cuuint32_t)box_outer};
  cuuint32_t estr[2] = {1u, 1u};
  CUresult r = enc(map, dtype == DGPT_F32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2,
                   const_cast<void*>(base), gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed with CUresult %d (inner=%lld outer=%lld ld=%lld)", (int)r,
              (long long)inner, (long long)outer, (long long)ld);
    return DGPT_E_ARG;
  }
  return DGPT_OK;
}

int make_tmap_bf16_2d(CUtensorMap* map, const void* base, int64_t inner, int64_t outer, int64_t ld, int box_outer) {
  return make_tmap_2d(map, base, DGPT_BF16, inner, outer, ld, 64, box_outer);
}

struct TcMaps {
  CUtensorMap a, b, d, r;
};

// persistent grid: one CTA per SM, or one per tile when there are fewer tiles
template <int BN, int A_MN, int B_MN, int EPI, int OBF, int CS = 0, int TM = 1>
static int launch_one(const TcMaps& m, const TcParams& p, int sms, cudaStream_t st) {
  using Cfg = TcCfg<BN, EPI, CS, TM>;
  auto kern = gemm_tc_kernel<BN, A_MN, B_MN, EPI, OBF, CS, TM>;
  static bool attr_done = false;
  if (!attr_done) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Cfg::kSmemBytes);
    if (e != cudaSuccess) {
      set_error("gemm_tc: cudaFuncSetAttribute(%zu B smem): %s", Cfg::kSmemBytes, cudaGetErrorString(e));
      return DGPT_E_LAUNCH;
    }
    attr_done = true;
  }
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)min(p.m_tiles * p.n_tiles * p.split_k, sms));
  cfg.blockDim = dim3(kThreads);
  cfg.dynamicSmemBytes = Cfg::kSmemBytes;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = pdl_enabled() ? 1 : 0;
  cudaError_t e = cudaLaunchKernelEx(&cfg, kern, m.a, m.b, m.d, m.r, p);
  if (e != cudaSuccess) {
    set_error("gemm_tc: launch: %s", cudaGetErrorString(e));
    return DGPT_E_LAUNCH;
  }
  return check_launch("gemm_tc");
}

int launch_gemm_tc(const dgpt_gemm_args* a, cudaStream_t st) {
  DGPT_REQUIRE(a->K > 0, "gemm(bf16): K must be positive");
  const int a_mn = a->a_major == DGPT_MAJOR_MN, b_mn = a->b_major == DGPT_MAJOR_MN;
  DGPT_REQUIRE(!(a_mn && !b_mn), "gemm(bf16): A MN-major with B K-major is not instantiated");
  // tile N: widest tile that still yields >= ~1 wave of CTAs
  int sms = dgpt_sm_count();
  if (sms <= 0) sms = 148;
  int m_tiles = ceil_div(a->M, TBM);
  // 128 x 256 tiles ingest 25 % fewer operand bytes per MMA cycle than 128 x 128; a ragged last column
  // tile (N = 1152 -> 4.5 tiles) costs less than that as soon as N >= 1024 (TMA zero-fills, the store clips)
  int BN = 256;
  // wgrads that carry a column sum (bias gradient): 256-column tiles when the output has few row tiles and wide rows
  // (FFN2: 384 x 1536) -- a 128 x 128 tile needs 64 operand bytes per 1 K MMA cycles where the SM ingests ~70 B/cycle,
  // a 128 x 256 tile 48; their single accumulator buffer costs nothing because a split-K CTA owns one tile.
  // (Runner._splits mirrors this rule when it picks the wgrad split count.)
  const bool cs_wide = a->a_colsum && a->N % 256 == 0 && a->N >= 512 && m_tiles < 8;
  if (a->N <= 128 || (a->N % 256 != 0 && a->N < 1024) || (a->a_colsum && !cs_wide)) BN = 128;
  if (BN == 256 && !cs_wide && m_tiles * ceil_div(a->N, 256) * (a->split_k > 1 ? a->split_k : 1) < sms) BN = 128;
  // 192-column tiles for N = 192, 384, 576, 960 (the model's N = 384 GEMMs): two tiles per row instead of three
  // (measured: ~5 % faster for the dgrad / wgrad GEMMs with >= 8 row tiles; slower with the residual epilogue, whose
  // three staging buffers per warp leave a 3-stage ring, and for small wgrads that would need > 20 K splits)
  // (the bit-mask epilogues are instantiated for 128- / 256-column tiles only)
  if (BN == 128 && a->N % 192 == 0 && a->N % 256 != 0 && a->N < 1024 && m_tiles >= 8 && !a->residual &&
      !a->relu_mask_in && !a->relu_mask_out)
    BN = 192;
  // Wave quantisation for the big-activation GEMMs (M >= 1024 rows, no split-K): a persistent grid of `sms` CTAs walks
  // m_tiles * n_tiles equal tiles, so 768 tiles on 148 SMs (N = 1536 with 256-column tiles) leave the last of 6 rounds
  // 81 % empty, and N = 1152 wastes half of every fifth column tile on top.  Pick the width with the best
  //   (useful columns / tiled columns) * (tiles / (rounds * sms)) * (tile-shape factor: 1.0 / 0.95 / 0.88 for 256 / 192 / 128,
  // measured: operand re-reads and per-tile bookkeeping).  FFN1 fwd / FFN2 dgrad (N = 1536): 192 (1024 tiles, 6.9 rounds);
  // QKV fwd (N = 1152): 128 (1152 tiles, 7.8 rounds).
  if (BN == 256 && !cs_wide && a->split_k <= 1 && m_tiles >= 8 && !a->residual && !a->a_colsum && a->N >= 1024) {
    auto score = [&](int bn, double shape) {
      const int nt = ceil_div(a->N, bn), tiles = m_tiles * nt, rounds = ceil_div(tiles, sms);
      return shape * ((double)a->N / (nt * bn)) * ((double)tiles / ((double)rounds * sms));
    };
    double best = score(256, 1.0);
    if (a->N % 192 == 0 && score(192, 0.95) > best) { best = score(192, 0.95); BN = 192; }
    if (score(128, 0.88) > best) BN = 128;
  }
  // 256-row CTA tiles (TM = 2: two M = 128 MMAs per k-step on one B stage, 1/3 fewer operand bytes per MMA cycle) for
  // the forward / dgrad GEMMs of the model's big activations: plain, bias + ReLU (+ mask) and mask-in epilogues with
  // bf16 output, no split-K, no residual (the TMA-fed residual path is a 128-row design).
  // Measured (profiles/r2_gemm_experiments.txt): 256-row tiles are 3 % faster for K >= 1024 (FFN1 / QKV dgrad) and
  // 10-20 % SLOWER for the K = 384 GEMMs, whose pace is set by the epilogue (single-buffered accumulators serialise it
  // with the mainloop): 256-row tiles only for K >= 1024.
  int TM = 1;
  if (a->K >= 1024 && !a_mn && a->M >= 1024 && a->d_dtype == DGPT_BF16 && !a->residual && !a->D2 && !a->relu_aux &&
      a->dropout_p == 0.f && a->split_k <= 1 && !a->accumulate && !a->a_colsum) {
    // tile width for 256-row tiles: 192 when it divides N (N = 384, 1152: no ragged column tile), else 256
    const int bn2 = (a->N % 192 == 0 && a->N % 256 != 0) ? 192 : (a->N >= 256 ? 256 : 0);
    // only the fast-path epilogues the model uses are instantiated for 256-row tiles (TMA-addressable bf16 output,
    // vector-aligned bias); everything else keeps 128-row tiles
    auto al16e = [](const void* q) { return ((uintptr_t)q & 15) == 0; };
    const bool fast_ok = al16e(a->D) && ((int64_t)a->ldd * 2) % 16 == 0 && a->N % 4 == 0 && (!a->bias || al16e(a->bias)) &&
                         ((!a->relu_mask_in && !a->relu_mask_out) || a->N % 64 == 0);
    const int e0 = (a->bias ? kEpiBias : 0) | (a->relu ? kEpiRelu : 0) | (a->relu_mask_in ? kEpiMaskIn : 0) |
                   (a->relu_mask_out ? kEpiMaskOut : 0);
    const bool inst = bn2 == 256 ? (b_mn ? (e0 == 0 || e0 == kEpiMaskIn)
                                         : (e0 == 0 || e0 == (kEpiBias | kEpiRelu) || e0 == (kEpiBias | kEpiRelu | kEpiMaskOut)))
                                 : (bn2 == 192 && e0 == 0);
    if (bn2 && fast_ok && inst) { TM = 2; BN = bn2; m_tiles = ceil_div(a->M, 2 * TBM); }
  }
  const int n_tiles = ceil_div(a->N, BN);
  TcParams p;
  p.M = a->M; p.N = a->N; p.K = a->K;
  p.m_tiles = m_tiles; p.n_tiles = n_tiles;
  p.kb_total = ceil_div(a->K, TBK);
  p.split_k = a->split_k > 1 ? min(a->split_k, p.kb_total) : 1;
  p.kb_per_split = ceil_div(p.kb_total, p.split_k);
  p.split_k = ceil_div(p.kb_total, p.kb_per_split);
  p.ep = make_epilogue(a);
  p.ep.atomic = p.split_k > 1;
  if (p.split_k > 1 && !a->accumulate) {
    cudaError_t e = cudaMemset2DAsync(a->D, (size_t)a->ldd * 4, 0, (size_t)a->N * 4, (size_t)a->M, st);
    if (e != cudaSuccess) { set_error("gemm_tc: memset: %s", cudaGetErrorString(e)); return DGPT_E_LAUNCH; }
  }
  auto al16 = [](const void* q) { return ((uintptr_t)q & 15) == 0; };
  p.vec_ok = (a->N % 4 == 0) && (!a->bias || al16(a->bias)) && (!a->residual || (al16(a->residual) && a->ldr % 4 == 0));
  p.mask_out = a->relu_mask_out;
  p.mask_in = a->relu_mask_in;
  p.a_colsum = a->a_colsum;
  p.probe = clock_probe_buffer();
  TcMaps mp;
  int rc;
  if (a_mn) rc = make_tmap_bf16_2d(&mp.a, a->A, a->M, a->K, a->lda, 64);
  else rc = make_tmap_bf16_2d(&mp.a, a->A, a->K, a->M, a->lda, TBM);
  if (rc) return rc;
  if (b_mn) rc = make_tmap_bf16_2d(&mp.b, a->B, a->N, a->K, a->ldb, 64);
  else rc = make_tmap_bf16_2d(&mp.b, a->B, a->K, a->N, a->ldb, BN);
  if (rc) return rc;
  // output through TMA when its pitch allows it (always true for the model's buffers)
  const int desz = a->d_dtype == DGPT_F32 ? 4 : 2;
  p.store_mode = kStoreDirect;
  if (al16(a->D) && ((int64_t)a->ldd * desz) % 16 == 0) {
    rc = make_tmap_2d(&mp.d, a->D, a->d_dtype, a->N, a->M, a->ldd, 128 / desz, 32);
    if (rc) return rc;
    p.store_mode = (p.ep.atomic || a->accumulate) ? kStoreTmaAdd : kStoreTma;
  } else {
    mp.d = mp.a;
  }
  mp.r = mp.a;

  // Epilogue specialisation: the combinations the model uses get their own (fast-path) instantiation, the
  // rest run the generic element-wise kernel.  Fast path needs TMA-addressable output, vector-aligned
  // operands, no second output, no saved-activation mask, and (bias / residual) no split-K.
  int epi = (a->bias ? kEpiBias : 0) | (a->relu ? kEpiRelu : 0) | (a->relu_aux ? kEpiAux : 0) |
            (a->dropout_p > 0.f ? kEpiDrop : 0) | (a->residual ? kEpiRes : 0) | (a->relu_mask_in ? kEpiMaskIn : 0) |
            (a->relu_mask_out ? kEpiMaskOut : 0);
  const int obf = a->d_dtype == DGPT_BF16 ? 1 : 0;
  if (a->relu_mask_in || a->relu_mask_out) {
    DGPT_REQUIRE(p.store_mode != kStoreDirect && p.vec_ok && !a->D2 && !a->relu_aux && a->N % 64 == 0 && obf && p.split_k == 1,
                 "gemm(bf16): relu_mask_in/out need a bf16, 16-byte aligned output with N %% 64 == 0 and no split-K");
    DGPT_REQUIRE(epi == kEpiMaskIn || epi == (kEpiBias | kEpiRelu | kEpiMaskOut),
                 "gemm(bf16): relu_mask_out goes with bias + ReLU only, relu_mask_in with a plain epilogue only");
  }
  DGPT_REQUIRE(!a->a_colsum || (a_mn && b_mn && p.store_mode != kStoreDirect && p.vec_ok && !a->D2),
               "gemm(bf16): a_colsum rides on MN-major (wgrad) GEMMs with a 16-byte aligned fp32 output");
  if (p.store_mode == kStoreDirect || !p.vec_ok || a->D2 || a->relu_aux) epi = -1;
  if (epi > 0 && (epi & (kEpiBias | kEpiRes)) && p.split_k > 1) epi = -1;
  if (epi >= 0 && (epi & kEpiRes)) {
    if ((BN != 128 && BN != 192) || obf) {
      epi = -1;  // the TMA-fed residual path is instantiated for 128- / 192-column tiles with fp32 output
    } else {
      DGPT_REQUIRE(a->ldr % 4 == 0, "gemm(bf16): residual pitch");
      if ((rc = make_tmap_2d(&mp.r, a->residual, DGPT_F32, a->N, a->M, a->ldr, 32, 32))) return rc;
    }
  }
#define TC_EPI(BN_, A_, B_, E_, O_) \
  if (epi == (E_) && obf == (O_)) return launch_one<BN_, A_, B_, (E_), O_>(mp, p, sms, st);
#define TC_DISPATCH(BN_)                                                              \
  if (BN == BN_) {                                                                    \
    if (!a_mn && !b_mn) {                                                             \
      TC_EPI(BN_, 0, 0, 0, 1)                                                         \
      if (BN_ == 128) { TC_EPI(128, 0, 0, kEpiBias, 0) }  /* lm_head: fp32 logits, N = 80 (full blocks fast) */ \
      TC_EPI(BN_, 0, 0, kEpiBias | kEpiRelu, 1)                                       \
      TC_EPI(BN_, 0, 0, kEpiBias | kEpiRelu | kEpiMaskOut, 1)                         \
      if (BN_ == 128) {                                                               \
        TC_EPI(128, 0, 0, kEpiBias | kEpiRes, 0)                                      \
        TC_EPI(128, 0, 0, kEpiBias | kEpiDrop | kEpiRes, 0)                           \
      }                                                                               \
      return launch_one<BN_, 0, 0, -1, 0>(mp, p, sms, st);                            \
    }                                                                                 \
    if (!a_mn && b_mn) {                                                              \
      TC_EPI(BN_, 0, 1, 0, 1)                                                         \
      TC_EPI(BN_, 0, 1, 0, 0)                                                         \
      TC_EPI(BN_, 0, 1, kEpiMaskIn, 1)                                                \
      return launch_one<BN_, 0, 1, -1, 0>(mp, p, sms, st);                            \
    }                                                                                 \
    if (a->a_colsum) {                                                                \
      DGPT_REQUIRE(epi == 0 && obf == 0, "gemm(bf16): a_colsum needs the plain fp32 wgrad form");   \
      return launch_one<BN_, 1, 1, 0, 0, 1>(mp, p, sms, st);                          \
    }                                                                                 \
    TC_EPI(BN_, 1, 1, 0, 0)                                                           \
    return launch_one<BN_, 1, 1, -1, 0>(mp, p, sms, st);                              \
  }
  if (TM == 2) {
#define TC_TM2(BN_, B_, E_) \
    if (BN == (BN_) && b_mn == (B_) && epi == (E_) && obf == 1) return launch_one<BN_, 0, B_, (E_), 1, 0, 2>(mp, p, sms, st);
    TC_TM2(256, 0, 0)
    TC_TM2(256, 0, kEpiBias | kEpiRelu | kEpiMaskOut)
    TC_TM2(256, 0, kEpiBias | kEpiRelu)
    TC_TM2(256, 1, 0)
    TC_TM2(256, 1, kEpiMaskIn)
    TC_TM2(192, 0, 0)
    TC_TM2(192, 1, 0)
#undef TC_TM2
    set_error("gemm_tc: internal: no 256-row instantiation for BN=%d b_mn=%d epi=%d", BN, b_mn, epi);
    return DGPT_E_ARG;
  }
  if (BN == 192) {  // the instantiations the N = 384 GEMMs of the model need, else generic
#define TC_192(A_, B_, E_, O_, C_) \
    if (a_mn == (A_) && b_mn == (B_) && epi == (E_) && obf == (O_) && (a->a_colsum != nullptr) == ((C_) != 0)) \
      return launch_one<192, A_, B_, (E_), O_, C_>(mp, p, sms, st);
    TC_192(0, 0, 0, 1, 0)
    TC_192(0, 0, kEpiBias | kEpiRelu, 1, 0)
    TC_192(0, 0, kEpiBias | kEpiRelu | kEpiMaskOut, 1, 0)
    TC_192(0, 1, kEpiMaskIn, 1, 0)
    TC_192(0, 1, 0, 1, 0)
    TC_192(0, 1, 0, 0, 0)
    TC_192(1, 1, 0, 0, 0)
    TC_192(1, 1, 0, 0, 1)
#undef TC_192
    DGPT_REQUIRE(!a->a_colsum, "gemm(bf16): a_colsum needs the plain fp32 wgrad form");
    if (!a_mn && !b_mn) return launch_one<192, 0, 0, -1, 0>(mp, p, sms, st);
    if (!a_mn && b_mn) return launch_one<192, 0, 1, -1, 0>(mp, p, sms, st);
    return launch_one<192, 1, 1, -1, 0>(mp, p, sms, st);
  }
  TC_DISPATCH(128)
  TC_DISPATCH(256)
#undef TC_DISPATCH
#undef TC_EPI
  set_error("gemm_tc: no tile configuration for N=%d", a->N);
  return DGPT_E_ARG;
}

}  // namespace dgpt
