// KV-cached generation kernels for sm_100a (tensor-mode weights: bf16 shadows, fp32 statistics).
//
// Replaces the reference's `generate` loop (src/model.py:611-636: full forward over the cropped window + softmax +
// torch.multinomial + torch.cat per token) while the window has not slid (SURVEY Q12):
//
//   decode_attn_kernel<WPU>   one new query per (sequence, head) against the cached keys / values: 1-8 warps per
//                             (b, h) with the keys split between them, 8 lanes per key row, online softmax over 32-key
//                             chunks -- the batch-1024 end of the sweep is bound by streaming the KV cache, so the kernel
//                             is built to keep HBM busy (16 x 16 B in flight per lane: the K and V rows of a chunk)
//   decode_persistent_kernel  small batches (<= 8 sequences): ONE launch generates every token of the in-window part.
//                             All layers of a token run as phases of a persistent grid (LayerNorm fused into the
//                             matrix-vector prologue, bias / ReLU / residual into its epilogue, KV append, attention,
//                             LM head, on-device sampling: warp_sample_row of sample.cuh) separated by cluster barriers;
//                             the 21.6 MB of bf16 weights stay L2-resident across tokens.  The launch-per-kernel path
//                             needs ~45 launches per token; this one needs none.
#include <cuda.h>
#include <stdlib.h>

#include "common.cuh"
#include "sample.cuh"

namespace dgpt {

static constexpr int kDecH = 64;      // head size
static constexpr int kDecMaxB = 8;    // sequences per persistent launch
static constexpr int kDecMaxL = 8;    // layers
static constexpr int kDecThreads = 256;

#ifndef DEC_LD
#define DEC_LD(p) __ldg(p)
#endif
__device__ __forceinline__ float bf16_lo(uint32_t w) { return __uint_as_float(w << 16); }
__device__ __forceinline__ float bf16_hi(uint32_t w) { return __uint_as_float(w & 0xFFFF0000u); }

// ---------------------------------------------------------------------------
// batched decode attention (any batch): WPU warps per (sequence, head), keys split between them
//
// Lane mapping: 8 lanes share one key (lane & 7 = which 16-byte chunk of its 128-byte row), 4 keys per warp
// instruction (lane >> 3).  A load instruction therefore touches 4 full 128-byte lines -- 4 L1 wavefronts -- where
// one-key-per-lane touched 32 lines with 16 bytes each (32 wavefronts: that version ran at the L1 wavefront rate,
// 2.5 TB/s of KV bytes, not at HBM speed).
// A warp walks its key range in chunks of 32 with an ONLINE softmax: the 8 K rows and the 8 V rows of a chunk are
// requested together (8 KB in flight per warp, one memory round trip per chunk instead of a score pass followed by
// a value pass), and the WPU partial (max, sum, output) triples of a (sequence, head) are merged through shared
// memory.  WPU (1 / 2 / 4 / 8) is chosen by the host: as many warps as it takes to fill the machine once, never more
// than there are 32-key chunks.  The previous version (a score pass into shared memory, then a value pass, 4 KB in
// flight per warp, 4 CTAs per SM = 1.3 waves at batch 1024) ran at 0.53-0.67 of HBM; this one at 0.86-0.93.
// ---------------------------------------------------------------------------
struct DecAttnP {
  const __nv_bfloat16 *q, *k, *v;
  __nv_bfloat16* o;
  int64_t q_bs, k_bs, k_rs, v_bs, v_rs, o_bs;
  int B, NH, nk;
  float scale;
};

__device__ __forceinline__ float dot8q(const uint4& w, const float (&q)[8]) {
  return q[0] * bf16_lo(w.x) + q[1] * bf16_hi(w.x) + q[2] * bf16_lo(w.y) + q[3] * bf16_hi(w.y) + q[4] * bf16_lo(w.z) +
         q[5] * bf16_hi(w.z) + q[6] * bf16_lo(w.w) + q[7] * bf16_hi(w.w);
}

template <int WPU>
__global__ void __launch_bounds__(kDecThreads, 2) decode_attn_kernel(DecAttnP p) {
  pdl_grid_sync();
  constexpr int kWarps = kDecThreads / 32, kUnits = kWarps / WPU;
  __shared__ float part_s[kWarps][kDecH + 2];  // per warp: running max, sum of exp, unnormalised output[64]
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int bh = blockIdx.x * kUnits + w / WPU, wi = w % WPU;
  const bool live = bh < p.B * p.NH;
  const int b = live ? bh / p.NH : 0, h = live ? bh % p.NH : 0;
  const int g = lane >> 3, c = lane & 7;
  const int nk = p.nk;
  const int per = ((nk + WPU - 1) / WPU + 3) & ~3;  // keys per warp
  const int j_lo = wi * per, j_hi = live ? min(nk, j_lo + per) : 0;
  float q[8];
  {
    const uint4 u = __ldg(reinterpret_cast<const uint4*>(p.q + b * p.q_bs + h * kDecH) + c);
    q[0] = bf16_lo(u.x) * p.scale; q[1] = bf16_hi(u.x) * p.scale; q[2] = bf16_lo(u.y) * p.scale; q[3] = bf16_hi(u.y) * p.scale;
    q[4] = bf16_lo(u.z) * p.scale; q[5] = bf16_hi(u.z) * p.scale; q[6] = bf16_lo(u.w) * p.scale; q[7] = bf16_hi(u.w) * p.scale;
  }
  const __nv_bfloat16* kb = p.k + b * p.k_bs + h * kDecH;
  const __nv_bfloat16* vb = p.v + b * p.v_bs + h * kDecH;
  float mx = -INFINITY, sum = 0.f;  // sum: this lane group's keys only (added over the 4 groups at the end)
  float o[8];
#pragma unroll
  for (int d = 0; d < 8; ++d) o[d] = 0.f;
  for (int j0 = j_lo; j0 < j_hi; j0 += 32) {
    uint4 kr[8], vr[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int j = j0 + i * 4 + g;
      kr[i] = (j < j_hi) ? DEC_LD(reinterpret_cast<const uint4*>(kb + (int64_t)j * p.k_rs) + c) : make_uint4(0u, 0u, 0u, 0u);
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int j = j0 + i * 4 + g;
      vr[i] = (j < j_hi) ? DEC_LD(reinterpret_cast<const uint4*>(vb + (int64_t)j * p.v_rs) + c) : make_uint4(0u, 0u, 0u, 0u);
    }
    float sc[8], cm = -INFINITY;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      float d = dot8q(kr[i], q);
      d += __shfl_xor_sync(0xffffffffu, d, 1);
      d += __shfl_xor_sync(0xffffffffu, d, 2);
      d += __shfl_xor_sync(0xffffffffu, d, 4);
      sc[i] = (j0 + i * 4 + g < j_hi) ? d : -INFINITY;
      cm = fmaxf(cm, sc[i]);
    }
    cm = fmaxf(cm, __shfl_xor_sync(0xffffffffu, cm, 8));
    cm = fmaxf(cm, __shfl_xor_sync(0xffffffffu, cm, 16));  // chunk maximum, warp-uniform (key j0 is always valid: finite)
    const float nm = fmaxf(mx, cm), rs = __expf(mx - nm);
    mx = nm;
    sum *= rs;
#pragma unroll
    for (int d = 0; d < 8; ++d) o[d] *= rs;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const float pj = __expf(sc[i] - nm);
      sum += pj;
      o[0] += pj * bf16_lo(vr[i].x); o[1] += pj * bf16_hi(vr[i].x); o[2] += pj * bf16_lo(vr[i].y); o[3] += pj * bf16_hi(vr[i].y);
      o[4] += pj * bf16_lo(vr[i].z); o[5] += pj * bf16_hi(vr[i].z); o[6] += pj * bf16_lo(vr[i].w); o[7] += pj * bf16_hi(vr[i].w);
    }
  }
  sum += __shfl_xor_sync(0xffffffffu, sum, 8);
  sum += __shfl_xor_sync(0xffffffffu, sum, 16);
#pragma unroll
  for (int d = 0; d < 8; ++d) {
    o[d] += __shfl_xor_sync(0xffffffffu, o[d], 8);
    o[d] += __shfl_xor_sync(0xffffffffu, o[d], 16);
  }
  if (WPU == 1) {
    if (g == 0 && live) {
      const float inv = 1.f / sum;
      __nv_bfloat162 a = __floats2bfloat162_rn(o[0] * inv, o[1] * inv), b2 = __floats2bfloat162_rn(o[2] * inv, o[3] * inv);
      __nv_bfloat162 c2 = __floats2bfloat162_rn(o[4] * inv, o[5] * inv), d2 = __floats2bfloat162_rn(o[6] * inv, o[7] * inv);
      uint4 out;
      out.x = *reinterpret_cast<uint32_t*>(&a); out.y = *reinterpret_cast<uint32_t*>(&b2);
      out.z = *reinterpret_cast<uint32_t*>(&c2); out.w = *reinterpret_cast<uint32_t*>(&d2);
      reinterpret_cast<uint4*>(p.o + b * p.o_bs + h * kDecH)[c] = out;
    }
    return;
  }
  // ---- merge the WPU partial results of this (sequence, head): warp wi == 0, lane -> output dims 2 lane, 2 lane + 1 ----
  if (lane == 0) { part_s[w][0] = mx; part_s[w][1] = sum; }
  if (g == 0) {
#pragma unroll
    for (int d = 0; d < 8; ++d) part_s[w][2 + c * 8 + d] = o[d];
  }
  __syncthreads();
  if (wi == 0 && live) {
    float M = -INFINITY;
#pragma unroll
    for (int u = 0; u < WPU; ++u) M = fmaxf(M, part_s[w + u][0]);
    float L = 0.f, a0 = 0.f, a1 = 0.f;
#pragma unroll
    for (int u = 0; u < WPU; ++u) {
      const float f = __expf(part_s[w + u][0] - M);  // a warp without keys holds (-inf, 0, 0): f = 0
      L += f * part_s[w + u][1];
      a0 += f * part_s[w + u][2 + 2 * lane];
      a1 += f * part_s[w + u][3 + 2 * lane];
    }
    const float inv = 1.f / L;
    reinterpret_cast<__nv_bfloat162*>(p.o + b * p.o_bs + h * kDecH)[lane] = __floats2bfloat162_rn(a0 * inv, a1 * inv);
  }
}

// ---------------------------------------------------------------------------
// persistent generation: one thread-block CLUSTER per group of <= 8 sequences
// ---------------------------------------------------------------------------
// The phases of a token (per layer: ln1 + QKV + KV append | attention | projection + residual | ln2 + FFN1 + ReLU |
// FFN2 + residual; then LM head | sampling) are separated by HARDWARE cluster barriers (barrier.cluster, ~0.2 us)
// instead of grid-wide atomics (~1.6 us measured), so the whole kernel is one cluster of 16 (or 8) CTAs per sequence
// group; several groups run side by side as independent clusters.  Every matrix-vector phase fetches ALL the weight
// rows its warp will need into registers BEFORE the barrier it waits on (the weights do not depend on the previous
// phase), so after the barrier a phase costs one L2 round trip for the activations plus the math.  Attention spreads
// the keys of one (sequence, head) over the threads of a CTA, so the KV rows of a position are fetched in one wave.
static constexpr int kPThreads = 256;        // threads per CTA (up to 255 registers each: the prefetched weights live there)
static constexpr int kPWarps = kPThreads / 32;
static constexpr int kPreMax = 24;           // 16-byte weight chunks a lane may hold across a barrier

struct DecLayerP {
  const __nv_bfloat16 *wqkv, *wproj, *w1, *w2;  // [3D, C], [C, D], [F, C], [C, F]  (nn.Linear layout, bf16 shadows)
  const float *ln1g, *ln1b, *ln2g, *ln2b, *bproj, *b1, *b2;
  __nv_bfloat16* cache;  // [B, ctx, 3D]: row (b, t) = the packed q | k | v of position t of sequence b
};

// layer table in constant memory (indexed with a run-time layer number: kernel parameters cannot be, the compiler
// would copy them to local memory, which every cluster barrier flushes from L1)
__constant__ DecLayerP c_dec_layers[kDecMaxL];

struct DecP {
  int nl;
  const float *tok, *pos;       // [V, C], [ctx, C]
  const __nv_bfloat16* wlm;     // [V, C]
  const float* blm;             // [V]
  int64_t* seq;                 // [ctx + 1, B] time-major token ids
  float *xa, *xb, *qbuf, *att, *hbuf, *logits;  // [B, C], [B, C], [B, D], [B, D], [B, F], [B, V] scratch
  int B, Bc, C, NH, F, V, ctx;  // Bc = sequences per cluster
  int t0, t1, t_sample;         // positions [t0, t1); tokens are sampled for t >= t_sample (earlier ones: prompt)
  int greedy;
  uint64_t seed;
  const uint64_t* seed_dev;
  const dgpt_sampling* sampling;  // NULL: plain multinomial
  float eps;
  unsigned long long* probe;    // DGPT_CLOCK_PROBE: phase stamps of the last position (cluster 0, CTA 0)
};

__device__ __forceinline__ uint32_t cluster_rank() { uint32_t r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ uint32_t cluster_size() { uint32_t r; asm volatile("mov.u32 %0, %%cluster_nctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ uint32_t cluster_id() { uint32_t r; asm volatile("mov.u32 %0, %%clusterid.x;" : "=r"(r)); return r; }
// cluster-wide barrier with release / acquire semantics: global-memory writes of every CTA before it are visible to
// every CTA after it (exchanged buffers are read with ld.global.cg, i.e. from L2, so no L1 line can be stale)
__device__ __forceinline__ void cluster_sync() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}

// store v into the same shared-memory slot of EVERY CTA of the cluster (distributed shared memory)
__device__ __forceinline__ void bcast_f32(float* local_slot, int cs, float v) {
  const uint32_t a = (uint32_t)__cvta_generic_to_shared(local_slot);
  for (int r = 0; r < cs; ++r) {
    uint32_t ra;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(ra) : "r"(a), "r"(r));
    asm volatile("st.shared::cluster.f32 [%0], %1;" ::"r"(ra), "f"(v) : "memory");
  }
}
__device__ __forceinline__ void st_rank_f32(float* local_slot, int rank, float v) {
  const uint32_t a = (uint32_t)__cvta_generic_to_shared(local_slot);
  uint32_t ra;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(ra) : "r"(a), "r"(rank));
  asm volatile("st.shared::cluster.f32 [%0], %1;" ::"r"(ra), "f"(v) : "memory");
}

// dst[b][0..K) = LayerNorm(src[b]) over rows held in THIS CTA's shared memory (K <= 512); one warp per row
__device__ __forceinline__ void ln_rows_smem(const float* src, const float* __restrict__ gamma, const float* __restrict__ beta,
                                             float* dst, int B, int K, float eps) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  for (int b = w; b < B; b += kPWarps) {
    const float4* r = reinterpret_cast<const float4*>(src + b * K);
    float4 v[4];
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int c = lane + 32 * i;
      v[i] = (c < (K >> 2)) ? r[c] : make_float4(0.f, 0.f, 0.f, 0.f);
      s += v[i].x + v[i].y + v[i].z + v[i].w;
    }
    const float mean = warp_sum(s) / (float)K;
    float q = 0.f;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      if (lane + 32 * i < (K >> 2)) {
        const float a = v[i].x - mean, b2 = v[i].y - mean, c2 = v[i].z - mean, d = v[i].w - mean;
        q += a * a + b2 * b2 + c2 * c2 + d * d;
      }
    }
    const float rstd = rsqrtf(warp_sum(q) / (float)K + eps);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int c = lane + 32 * i;
      if (c < (K >> 2)) {
        const float4 g = __ldg(reinterpret_cast<const float4*>(gamma) + c), be = __ldg(reinterpret_cast<const float4*>(beta) + c);
        float4 o;
        o.x = (v[i].x - mean) * rstd * g.x + be.x;
        o.y = (v[i].y - mean) * rstd * g.y + be.y;
        o.z = (v[i].z - mean) * rstd * g.z + be.z;
        o.w = (v[i].w - mean) * rstd * g.w + be.w;
        *reinterpret_cast<float4*>(dst + b * K + c * 4) = o;
      }
    }
  }
  __syncthreads();
}

// Weight rows of one matrix-vector phase, distributed over the warps of the cluster: warp gw owns rows gw, gw + nw, ...
// KC = 16-byte weight chunks per lane per row (2 for K <= 512, 6 for K <= 1536); up to 16 rows per warp, all fetched
// into registers before the barrier the phase waits on (kPreMax chunks; this model's shapes on a 16-CTA cluster fit).
// (accumulators must only ever be indexed with compile-time constants -- a run-time index would move the array to
// local memory and turn every multiply-add into a dependent load / store pair)
struct WPre {
  uint4 w[kPreMax];
  float bias;  // lane i: bias of this warp's i-th row
};
template <int KC>
__device__ __forceinline__ void gemv_prefetch_t(WPre& pre, const __nv_bfloat16* __restrict__ W, const float* __restrict__ bias,
                                                int N, int K, int gw, int nw) {
  const int lane = threadIdx.x & 31;
  pre.bias = (bias && gw + lane * nw < N) ? __ldg(bias + gw + lane * nw) : 0.f;
#pragma unroll
  for (int i = 0; i < kPreMax / KC; ++i) {
    const int n = gw + i * nw;
    if (n < N) {
      const uint4* wr = reinterpret_cast<const uint4*>(W + (int64_t)n * K);
#pragma unroll
      for (int cc = 0; cc < KC; ++cc)
        if (lane + 32 * cc < (K >> 3)) pre.w[i * KC + cc] = __ldg(wr + lane + 32 * cc);
    }
  }
}
__device__ __forceinline__ void gemv_prefetch(WPre& pre, const __nv_bfloat16* __restrict__ W, const float* __restrict__ bias,
                                              int N, int K, int gw, int nw) {
  if (K <= 512) gemv_prefetch_t<2>(pre, W, bias, N, K, gw, nw);
  else gemv_prefetch_t<6>(pre, W, bias, N, K, gw, nw);
}

__device__ __forceinline__ float dot8(const uint4& wv, const float* x) {
  const float4 x0 = *reinterpret_cast<const float4*>(x);
  const float4 x1 = *reinterpret_cast<const float4*>(x + 4);
  return bf16_lo(wv.x) * x0.x + bf16_hi(wv.x) * x0.y + bf16_lo(wv.y) * x0.z + bf16_hi(wv.y) * x0.w + bf16_lo(wv.z) * x1.x +
         bf16_hi(wv.z) * x1.y + bf16_lo(wv.w) * x1.z + bf16_hi(wv.w) * x1.w;
}

// 16 per-lane partial sums (one per row) -> lane l holds the warp-wide total of row (l & 15): a halving butterfly
// (16 shuffles) instead of 16 full reductions (80 shuffles)
__device__ __forceinline__ float rows16_reduce(float (&v)[16], int lane) {
#pragma unroll
  for (int step = 0; step < 4; ++step) {
    const int mk = 8 >> step, n = 8 >> step;  // lane mask 8, 4, 2, 1; values kept 8, 4, 2, 1
    const bool upper = (lane & mk) != 0;
#pragma unroll
    for (int d = 0; d < n; ++d) {
      const float mine = upper ? v[d + n] : v[d];
      const float send = upper ? v[d] : v[d + n];
      v[d] = mine + __shfl_xor_sync(0xffffffffu, send, mk);
    }
  }
  return v[0] + __shfl_xor_sync(0xffffffffu, v[0], 16);
}

// y[b][n] = sum_k x[b][k] * W[n][k] for this warp's rows n = gw + i * nw (i < 16): x in shared memory ([B][K]);
// lane i (< 16) calls emit(b, n, total, bias_n) for its row -- the rows of a warp are emitted in parallel
template <int BM, int KC, typename Emit>
__device__ __forceinline__ void gemv_rows_t(const __nv_bfloat16* __restrict__ W, const WPre& pre, const float* x, int N, int K,
                                            int B, int gw, int nw, Emit emit) {
  const int lane = threadIdx.x & 31;
  constexpr int R = kPreMax / KC;  // rows whose weights are in registers (<= 16)
  static_assert(R <= 16, "at most 16 rows per warp");
  const int my_n = gw + (lane & 15) * nw;
#pragma unroll
  for (int b = 0; b < BM; ++b) {
    if (b < B) {
      float part[16];
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        part[i] = 0.f;
        if (i < R && gw + i * nw < N) {
#pragma unroll
          for (int cc = 0; cc < KC; ++cc)
            if (lane + 32 * cc < (K >> 3)) part[i] += dot8(pre.w[i * KC + cc], x + b * K + (lane + 32 * cc) * 8);
        }
      }
      const float tot = rows16_reduce(part, lane);
      if (lane < R && my_n < N) emit(b, my_n, tot, pre.bias);
    }
  }
}
template <int BM, typename Emit>
__device__ __forceinline__ void gemv_rows(const __nv_bfloat16* __restrict__ W, const WPre& pre, const float* x, int N, int K, int B,
                                          int gw, int nw, Emit emit) {
  if (K <= 512) gemv_rows_t<BM, 2>(W, pre, x, N, K, B, gw, nw, emit);
  else gemv_rows_t<BM, 6>(W, pre, x, N, K, B, gw, nw, emit);
}

// One (sequence, head) handled by a whole CTA: thread j owns key j (nk <= 256 <= kPThreads), so every K / V row of
// the position is fetched in one wave of 16-byte loads; q comes from shared memory (qs), the result goes to out[64].
__device__ __forceinline__ void cta_attend(const float* qs, float* red, const __nv_bfloat16* __restrict__ kb,
                                           const __nv_bfloat16* __restrict__ vb, int64_t rs, int nk, float scale,
                                           float* __restrict__ out) {
  const int j = threadIdx.x, lane = j & 31, w = j >> 5;
  const int nwk = (nk + 31) >> 5;  // warps that own keys
  float sc = -INFINITY;
  uint4 wv[8];
  if (j < nk) {
    const uint4* kr = reinterpret_cast<const uint4*>(kb + (int64_t)j * rs);
#pragma unroll
    for (int c = 0; c < 8; ++c) wv[c] = __ldcg(kr + c);
    float acc = 0.f;
#pragma unroll
    for (int c = 0; c < 8; ++c) {
      const uint32_t u[4] = {wv[c].x, wv[c].y, wv[c].z, wv[c].w};
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        acc = fmaf(qs[c * 8 + 2 * e], bf16_lo(u[e]), acc);
        acc = fmaf(qs[c * 8 + 2 * e + 1], bf16_hi(u[e]), acc);
      }
    }
    sc = acc * scale;
    const uint4* vr = reinterpret_cast<const uint4*>(vb + (int64_t)j * rs);  // values requested before the reductions
#pragma unroll
    for (int c = 0; c < 8; ++c) wv[c] = __ldcg(vr + c);
  }
  // block max / sum over the key-owning warps (red[0..15] max, red[16..31] sum)
  float m = warp_max(sc);
  if (lane == 0) red[w] = m;
  __syncthreads();
  m = red[0];
  for (int i = 1; i < nwk; ++i) m = fmaxf(m, red[i]);
  const float e = (j < nk) ? __expf(sc - m) : 0.f;
  const float ssum = warp_sum(e);
  if (lane == 0) red[16 + w] = ssum;
  __syncthreads();
  float tot = 0.f;
  for (int i = 0; i < nwk; ++i) tot += red[16 + i];
  const float pj = e / tot;
  // weighted values: per-warp butterfly (lane l ends with dims 2 l, 2 l + 1 of its 32 keys), then across warps
  if (w < nwk) {
    float o[kDecH];
#pragma unroll
    for (int c = 0; c < 8; ++c) {
      const uint32_t u[4] = {wv[c].x, wv[c].y, wv[c].z, wv[c].w};
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        o[c * 8 + 2 * q] = (j < nk) ? pj * bf16_lo(u[q]) : 0.f;
        o[c * 8 + 2 * q + 1] = (j < nk) ? pj * bf16_hi(u[q]) : 0.f;
      }
    }
#pragma unroll
    for (int step = 0; step < 5; ++step) {
      const int mk = 16 >> step, n = kDecH >> (step + 1);
      const bool upper = (lane & mk) != 0;
#pragma unroll
      for (int d = 0; d < n; ++d) {
        const float mine = upper ? o[d + n] : o[d];
        const float send = upper ? o[d] : o[d + n];
        o[d] = mine + __shfl_xor_sync(0xffffffffu, send, mk);
      }
    }
    red[32 + w * kDecH + 2 * lane] = o[0];
    red[32 + w * kDecH + 2 * lane + 1] = o[1];
  }
  __syncthreads();
  if (j < kDecH) {
    float a = 0.f;
    for (int i = 0; i < nwk; ++i) a += red[32 + i * kDecH + j];
    out[j] = a;
  }
  __syncthreads();  // red / qs may be reused
}

template <int BM>
__global__ void __launch_bounds__(kPThreads, 1) decode_persistent_kernel(DecP p) {
  extern __shared__ __align__(16) float smem_f[];
  const int C = p.C, D = p.NH * kDecH, F = p.F, V = p.V;
  // every CTA of the cluster holds a full copy of the activations of the cluster's sequences (peers write them
  // through distributed shared memory), so a phase never waits for an L2 round trip on its inputs
  float* xa = smem_f;                 // [BM][C] residual stream (layer input / output)
  float* xb = xa + BM * C;            // [BM][C] after the attention branch
  float* xn = xb + BM * C;            // [BM][C] LayerNorm output (local)
  float* at = xn + BM * C;            // [BM][D] attention output
  float* hh = at + BM * D;            // [BM][F] FFN hidden activation
  float* lg = hh + BM * F;            // [BM][V] logits (only rank 0's copy is written)
  float* red = lg + BM * V;           // [32 + 8 * 64] attention reductions
  float* qs = red + 32 + 8 * kDecH;   // [64] query of the (sequence, head) in flight
  float* ao = qs + kDecH;             // [64] attention output of it
  float* ss = ao + kDecH;             // [4] sampling settings (dgpt_sampling), loaded once
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int cr = (int)cluster_rank(), cs = (int)cluster_size(), cid = (int)cluster_id();
  const int gw = cr * kPWarps + w, nw = cs * kPWarps;  // warp index / count inside the cluster
  const int b0 = cid * p.Bc;
  const int B = min(p.Bc, p.B - b0);  // sequences of this cluster (whole clusters without work exit together)
  if (B <= 0) return;
  float* qbuf = p.qbuf + (int64_t)b0 * D;
  const float scale = rsqrtf((float)kDecH);
  uint64_t seed = p.seed;
  if (p.seed_dev) seed += *p.seed_dev;
  if (threadIdx.x < 3)  // temperature, top_k (bits), top_p; NULL: 1, 0, 1
    ss[threadIdx.x] = p.sampling ? reinterpret_cast<const float*>(p.sampling)[threadIdx.x] : (threadIdx.x == 1 ? 0.f : 1.f);
  WPre pre;
  gemv_prefetch(pre, c_dec_layers[0].wqkv, nullptr, 3 * D, C, gw, nw);
  cluster_sync();  // every CTA of the cluster is running before anyone writes into a peer's shared memory
  int stamp_i = 4;
#define DTS() do { if (p.probe && blockIdx.x == 0 && threadIdx.x == 0 && t == p.t1 - 1 && stamp_i < 64) p.probe[stamp_i++] = (unsigned long long)clock64(); } while (0)

  for (int t = p.t0; t < p.t1; ++t) {
    DTS();
    // ---- embedding: x = tok[seq[t]] + pos[t]  (src/model.py:595-597), computed by every CTA for itself ----
    for (int i = threadIdx.x; i < B * C; i += kPThreads) {
      const int b = i / C, c = i - b * C;
      xa[i] = p.tok[__ldcg(p.seq + (int64_t)t * p.B + b0 + b) * C + c] + p.pos[(int64_t)t * C + c];
    }
    __syncthreads();
    for (int l = 0; l < p.nl; ++l) {
      const DecLayerP& L = c_dec_layers[l];
      __nv_bfloat16* row = L.cache + ((int64_t)b0 * p.ctx + t) * 3 * D;  // + b * ctx * 3D per sequence
      // ---- ln1 + packed QKV projection; q | k | v of position t appended to the cache (global: attention reads it) ----
      ln_rows_smem(xa, L.ln1g, L.ln1b, xn, B, C, p.eps);
      gemv_rows<BM>(L.wqkv, pre, xn, 3 * D, C, B, gw, nw, [&](int b, int n, float v, float) {
        row[(int64_t)b * p.ctx * 3 * D + n] = __float2bfloat16_rn(v);
        if (n < D) qbuf[b * D + n] = v;
      });
      cluster_sync();
      DTS();
      // ---- attention over the t + 1 cached positions: one CTA per (sequence, head), threads over keys ----
      for (int bh = cr; bh < B * p.NH; bh += cs) {
        const int b = bh / p.NH, h = bh % p.NH;
        if (threadIdx.x < kDecH) qs[threadIdx.x] = __ldcg(qbuf + b * D + h * kDecH + threadIdx.x);
        __syncthreads();
        const __nv_bfloat16* kb = L.cache + (int64_t)(b0 + b) * p.ctx * 3 * D + D + h * kDecH;
        cta_attend(qs, red, kb, kb + D, (int64_t)3 * D, t + 1, scale, ao);
        if (threadIdx.x < kDecH) bcast_f32(at + b * D + h * kDecH + threadIdx.x, cs, ao[threadIdx.x]);
        __syncthreads();
      }
      gemv_prefetch(pre, L.wproj, L.bproj, C, D, gw, nw);
      cluster_sync();
      DTS();
      // ---- output projection + bias + residual ----
#define DTS2(k) do { if (p.probe && blockIdx.x == 0 && threadIdx.x == 0 && t == p.t1 - 1 && l == 1) p.probe[48 + (k)] = (unsigned long long)clock64(); } while (0)
      DTS2(0);
      gemv_rows<BM>(L.wproj, pre, at, C, D, B, gw, nw, [&](int b, int n, float v, float bn) {
        bcast_f32(xb + b * C + n, cs, xa[b * C + n] + bn + v);
      });
      DTS2(1);
      gemv_prefetch(pre, L.w1, L.b1, F, C, gw, nw);
      DTS2(2);
      asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
      DTS2(3);
      asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
      DTS2(4);
      DTS();
      // ---- ln2 + FFN1 + bias + ReLU ----
      ln_rows_smem(xb, L.ln2g, L.ln2b, xn, B, C, p.eps);
      gemv_rows<BM>(L.w1, pre, xn, F, C, B, gw, nw, [&](int b, int n, float v, float bn) {
        bcast_f32(hh + b * F + n, cs, fmaxf(v + bn, 0.f));
      });
      gemv_prefetch(pre, L.w2, L.b2, C, F, gw, nw);
      cluster_sync();
      DTS();
      // ---- FFN2 + bias + residual ----
      gemv_rows<BM>(L.w2, pre, hh, C, F, B, gw, nw, [&](int b, int n, float v, float bn) {
        bcast_f32(xa + b * C + n, cs, xb[b * C + n] + bn + v);
      });
      if (l + 1 < p.nl) gemv_prefetch(pre, c_dec_layers[l + 1].wqkv, nullptr, 3 * D, C, gw, nw);
      else if (t >= p.t_sample) gemv_prefetch(pre, p.wlm, p.blm, V, C, gw, nw);
      else gemv_prefetch(pre, c_dec_layers[0].wqkv, nullptr, 3 * D, C, gw, nw);
      cluster_sync();
      DTS();
    }
    if (t < p.t_sample) continue;  // prompt position: only the cache was needed
    // ---- LM head (ln_f is NOT applied, like the reference: src/model.py:598-599); logits go to rank 0 ----
    gemv_rows<BM>(p.wlm, pre, xa, V, C, B, gw, nw, [&](int b, int n, float v, float bn) { st_rank_f32(lg + b * V + n, 0, v + bn); });
    gemv_prefetch(pre, c_dec_layers[0].wqkv, nullptr, 3 * D, C, gw, nw);
    cluster_sync();
    DTS();
    // ---- next token: warp_sample_row (sample.cuh) with u = philox(seed, t, b), the same rule and stream as dgpt_sample ----
    if (cr == 0) {
      const dgpt_sampling sp{ss[0], __float_as_int(ss[1]), ss[2]};
      for (int b = w; b < B; b += kPWarps) {
        const int choice = warp_sample_row(lg + b * V, V, p.greedy != 0, sp, (uint32_t)(b0 + b), (uint32_t)t, seed);
        if (lane == 0) p.seq[(int64_t)(t + 1) * p.B + b0 + b] = (int64_t)choice;
      }
    }
    cluster_sync();  // the sampled tokens (global memory) are visible to every CTA's next embedding lookup
  }
  cluster_sync();  // no CTA exits while a peer may still write into its shared memory
}

// cluster <= 0: the launch's default, 16 CTAs (DGPT_DECODE_CLUSTER overrides it; read once per process)
static int decode_cluster_size(int cluster) {
  if (cluster > 0) return cluster;
  static int env_cluster = -1;
  if (env_cluster < 0) { const char* e = getenv("DGPT_DECODE_CLUSTER"); env_cluster = e ? atoi(e) : 0; }
  return env_cluster > 0 ? env_cluster : 16;
}

// The shapes decode_persistent_kernel handles: the one rule behind dgpt_decode_persistent_supported and the launch.
// report: say why a shape is refused (dgpt_last_error).
static bool decode_persistent_shape_ok(int B, int nl, int C, int NH, int H, int F, int V, int ctx, int cluster, bool report) {
#define DEC_GATE(cond, ...) do { if (!(cond)) { if (report) set_error(__VA_ARGS__); return false; } } while (0)
  // ln_rows_smem holds a row in 4 float4 per lane (C <= 512); the 6-chunk matrix-vector form reads K <= 1536;
  // cta_attend gives each cached key a thread of its own (context <= 256)
  DEC_GATE(H == kDecH && B >= 1 && nl >= 1 && nl <= kDecMaxL && NH >= 1 && V >= 1 && C >= 8 && F >= 8 && C % 8 == 0 &&
               F % 8 == 0 && ctx >= 1 && ctx <= 256 && C <= 512 && F <= 1536 && NH * kDecH <= 1536,
           "decode_persistent: head size 64, <= 8 layers, C <= 512 and F <= 1536 multiples of 8, context <= 256 "
           "(H=%d layers=%d C=%d F=%d ctx=%d)", H, nl, C, F, ctx);
  cluster = decode_cluster_size(cluster);
  DEC_GATE(cluster == 16 || cluster == 8 || cluster == 4, "decode_persistent: cluster size %d (4, 8 or 16)", cluster);
  {
    // every weight row of a phase must fit the per-warp register budget: 12 rows of K <= 512, 4 rows of K <= 1536
    const int nwarps = cluster * kPWarps, D3 = 3 * NH * kDecH;
    const int r_c = C <= 512 ? 12 : 4, r_f = F <= 512 ? 12 : 4, r_d = NH * kDecH <= 512 ? 12 : 4;
    DEC_GATE(D3 <= r_c * nwarps && F <= r_c * nwarps && V <= r_c * nwarps && C <= r_d * nwarps && C <= r_f * nwarps,
             "decode_persistent: model too wide for a cluster of %d CTAs (3D=%d F=%d C=%d V=%d)", cluster, D3, F, C, V);
  }
  DEC_GATE(B <= kDecMaxB, "decode_persistent: batch %d > %d (use the launch-per-kernel path)", B, kDecMaxB);
#undef DEC_GATE
  return true;
}

}  // namespace dgpt

using namespace dgpt;

extern "C" {

int dgpt_decode_attn(const void* q, const void* k, const void* v, void* o, int64_t q_bs, int64_t k_bs, int64_t k_rs,
                     int64_t v_bs, int64_t v_rs, int64_t o_bs, int B, int NH, int H, int nk, float scale, void* stream) {
  DGPT_DEVICE_OR_RETURN();
  DGPT_REQUIRE(H == kDecH && nk >= 1 && nk <= 256, "decode_attn: head size 64 and 1 <= keys <= 256 (H=%d keys=%d)", H, nk);
  auto al = [](const void* ptr, int64_t a, int64_t b) { return ((uintptr_t)ptr & 15) == 0 && a % 8 == 0 && b % 8 == 0; };
  DGPT_REQUIRE(al(k, k_bs, k_rs) && al(v, v_bs, v_rs) && ((uintptr_t)q & 15) == 0 && ((uintptr_t)o & 15) == 0 && q_bs % 8 == 0 && o_bs % 8 == 0,
               "decode_attn: operands must be 16-byte aligned with strides that are multiples of 8 elements");
  if (B == 0) return DGPT_OK;
  DecAttnP p;
  p.q = (const __nv_bfloat16*)q; p.k = (const __nv_bfloat16*)k; p.v = (const __nv_bfloat16*)v; p.o = (__nv_bfloat16*)o;
  p.q_bs = q_bs; p.k_bs = k_bs; p.k_rs = k_rs; p.v_bs = v_bs; p.v_rs = v_rs; p.o_bs = o_bs;
  p.B = B; p.NH = NH; p.nk = nk; p.scale = scale;
  const int64_t units = (int64_t)B * NH;
  static int force = -1;  // DGPT_DECODE_WPU=1|2|4|8 pins the warps per (sequence, head) (experiments)
  if (force < 0) { const char* e = getenv("DGPT_DECODE_WPU"); force = e ? atoi(e) : 0; }
  // enough warps for one full wave (2 CTAs of 8 warps per SM), but never more warps than 32-key chunks: at batch 1024
  // one warp per (sequence, head) streams at 0.86-0.93 of the HBM peak and splitting only adds near-empty CTAs; at batch
  // 64 the 384 (sequence, head) pairs need 8 warps each to cover the machine (profiles/r2_decode.txt)
  const int cap = nk <= 32 ? 1 : nk <= 64 ? 2 : nk <= 128 ? 4 : 8;
  int need = 1;
  while (need < 8 && units * need < (int64_t)dgpt_sm_count() * 16) need *= 2;
  const int wpu = force ? force : need < cap ? need : cap;
  constexpr int kW = kDecThreads / 32;
  switch (wpu) {
    case 1: launch_pdl(decode_attn_kernel<1>, dim3(ceil_div(units, kW)), dim3(kDecThreads), 0, (cudaStream_t)stream, p); break;
    case 2: launch_pdl(decode_attn_kernel<2>, dim3(ceil_div(units, kW / 2)), dim3(kDecThreads), 0, (cudaStream_t)stream, p); break;
    case 4: launch_pdl(decode_attn_kernel<4>, dim3(ceil_div(units, kW / 4)), dim3(kDecThreads), 0, (cudaStream_t)stream, p); break;
    default: launch_pdl(decode_attn_kernel<8>, dim3(units), dim3(kDecThreads), 0, (cudaStream_t)stream, p); break;
  }
  return check_launch("decode_attn");
}

// layers: host array of nl x 12 device pointers in DecLayerP order (wqkv, wproj, w1, w2, ln1g, ln1b, ln2g, ln2b, bproj,
// b1, b2, cache); scratch: device fp32 buffer of dgpt_decode_persistent_scratch_floats() floats + 1 barrier word (the
// caller zeroes the LAST 4 bytes before every call); seq: [ctx + 1, B] int64, positions <= t0 (and the prompt) filled.
int64_t dgpt_decode_persistent_scratch_floats(int B, int C, int NH, int F, int V) {
  return (int64_t)B * (2 * C + 2 * NH * kDecH + F + V) + 4;
}

/* largest batch the persistent decoder is used for.  Above it the launch-per-kernel path (tcgen05 GEMMs on the
 * M = batch rows + the KV-streaming attention kernel) is faster: measured crossover between 8 and 16 sequences. */
int dgpt_decode_persistent_max_batch(void) { return kDecMaxB; }

int dgpt_decode_persistent_supported(int B, int nl, int C, int NH, int H, int F, int V, int ctx, int cluster) {
  return decode_persistent_shape_ok(B, nl, C, NH, H, F, V, ctx, cluster, false) ? 1 : 0;
}

int dgpt_decode_persistent_ex(const void* const* layers, int nl, const float* tok, const float* pos, const void* wlm,
                              const float* blm, int64_t* seq, float* scratch, int B, int C, int NH, int H, int F, int V,
                              int ctx, int t0, int t1, int t_sample, int greedy, uint64_t seed, const uint64_t* seed_dev,
                              const dgpt_sampling* sampling, int cluster, void* stream) {
  DGPT_DEVICE_OR_RETURN();
  DGPT_REQUIRE(layers && tok && pos && wlm && seq && scratch, "decode_persistent: NULL argument");
  if (!decode_persistent_shape_ok(B, nl, C, NH, H, F, V, ctx, cluster, true)) return DGPT_E_ARG;
  DGPT_REQUIRE(0 <= t0 && t0 <= t1 && t1 <= ctx, "decode_persistent: positions [%d, %d) outside the context %d", t0, t1, ctx);
  if (t0 == t1) return DGPT_OK;
  cluster = decode_cluster_size(cluster);
  // one cluster per sequence while the clusters can all be resident at once (16 CTAs of one cluster need 16 SMs of
  // ONE GPC: 4 co-resident clusters measured on B200), else several sequences per cluster
  static int env_nc = -1;
  if (env_nc < 0) { const char* e = getenv("DGPT_DECODE_CLUSTERS"); env_nc = e ? atoi(e) : 0; }
  const int max_clusters = env_nc > 0 ? env_nc : 4;
  const int nclusters = min(B, max_clusters);
  const int Bc = ceil_div(B, nclusters);
  DecP p;
  static DecLayerP host_layers[kDecMaxL];  // (static: the async copy below may read it after this call returns)
  for (int l = 0; l < nl; ++l) {
    const void* const* q = layers + l * 12;
    DecLayerP& L = host_layers[l];
    L.wqkv = (const __nv_bfloat16*)q[0]; L.wproj = (const __nv_bfloat16*)q[1]; L.w1 = (const __nv_bfloat16*)q[2];
    L.w2 = (const __nv_bfloat16*)q[3];
    L.ln1g = (const float*)q[4]; L.ln1b = (const float*)q[5]; L.ln2g = (const float*)q[6]; L.ln2b = (const float*)q[7];
    L.bproj = (const float*)q[8]; L.b1 = (const float*)q[9]; L.b2 = (const float*)q[10];
    L.cache = (__nv_bfloat16*)q[11];
    for (int i = 0; i < 12; ++i) DGPT_REQUIRE(q[i] != nullptr, "decode_persistent: layer %d pointer %d is NULL", l, i);
  }
  {
    cudaError_t e = cudaMemcpyToSymbolAsync(c_dec_layers, host_layers, sizeof(DecLayerP) * nl, 0, cudaMemcpyHostToDevice,
                                            (cudaStream_t)stream);
    if (e != cudaSuccess) { set_error("decode_persistent: layer table upload: %s", cudaGetErrorString(e)); return DGPT_E_LAUNCH; }
  }
  const int D = NH * kDecH;
  p.nl = nl; p.tok = tok; p.pos = pos; p.wlm = (const __nv_bfloat16*)wlm; p.blm = blm; p.seq = seq;
  float* s = scratch;
  p.xa = s; s += (int64_t)B * C;
  p.xb = s; s += (int64_t)B * C;
  p.qbuf = s; s += (int64_t)B * D;
  p.att = s; s += (int64_t)B * D;
  p.hbuf = s; s += (int64_t)B * F;
  p.logits = s; s += (int64_t)B * V;
  p.B = B; p.Bc = Bc; p.C = C; p.NH = NH; p.F = F; p.V = V; p.ctx = ctx; p.t0 = t0; p.t1 = t1; p.t_sample = t_sample;
  p.greedy = greedy; p.seed = seed; p.seed_dev = seed_dev; p.sampling = sampling; p.eps = 1e-5f;
  p.probe = clock_probe_buffer();
  const int bm = Bc <= 1 ? 1 : Bc <= 2 ? 2 : Bc <= 4 ? 4 : 8;
  const size_t smem = ((size_t)bm * (3 * C + D + F + V) + 32 + 8 * kDecH + 2 * kDecH + 4) * sizeof(float);
  auto kern = bm == 1 ? decode_persistent_kernel<1> : bm == 2 ? decode_persistent_kernel<2>
              : bm == 4 ? decode_persistent_kernel<4> : decode_persistent_kernel<8>;
  static size_t attr_bytes[4] = {0, 0, 0, 0};
  static bool np_done[4] = {false, false, false, false};
  const int ki = bm == 1 ? 0 : bm == 2 ? 1 : bm == 4 ? 2 : 3;
  if (smem > 48 * 1024 && smem > attr_bytes[ki]) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) { set_error("decode_persistent: smem attribute: %s", cudaGetErrorString(e)); return DGPT_E_LAUNCH; }
    attr_bytes[ki] = smem;
  }
  if (!np_done[ki]) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
    if (e != cudaSuccess) { set_error("decode_persistent: non-portable cluster attribute: %s", cudaGetErrorString(e)); return DGPT_E_LAUNCH; }
    np_done[ki] = true;
  }
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)(nclusters * cluster));
  cfg.blockDim = dim3(kPThreads);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = (cudaStream_t)stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = (unsigned)cluster;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  cudaError_t e = cudaLaunchKernelEx(&cfg, kern, p);
  if (e != cudaSuccess) {
    set_error("decode_persistent: launch (cluster of %d): %s", cluster, cudaGetErrorString(e));
    return DGPT_E_LAUNCH;
  }
  return check_launch("decode_persistent");
}

int dgpt_decode_persistent(const void* const* layers, int nl, const float* tok, const float* pos, const void* wlm,
                           const float* blm, int64_t* seq, float* scratch, int B, int C, int NH, int H, int F, int V, int ctx,
                           int t0, int t1, int t_sample, int greedy, uint64_t seed, const uint64_t* seed_dev, int cluster,
                           void* stream) {
  return dgpt_decode_persistent_ex(layers, nl, tok, pos, wlm, blm, seq, scratch, B, C, NH, H, F, V, ctx, t0, t1, t_sample,
                                   greedy, seed, seed_dev, nullptr, cluster, stream);
}

}  // extern "C"
