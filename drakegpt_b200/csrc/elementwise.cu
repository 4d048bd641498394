// HBM-bound kernels of the training step: embedding gather/scatter, LayerNorm
// forward/backward (+fused residual-grad add and dropout-masked bf16 copy),
// cross-entropy forward+backward, flat AdamW, dropout/cast, column sums and the
// on-device sampler.  All are grid-sized in multiples of the SM count or one
// warp per row with float4 accesses; none allocates or synchronises.
#include "common.cuh"
#include "ptx.cuh"
#include "sample.cuh"

namespace dgpt {

// SM count of the current device (grid sizing; 148 on B200)
#define kSMs (dgpt_sm_count())

// ---------------------------------------------------------------------------
// dropout_scale / cast
// ---------------------------------------------------------------------------
template <typename OutT>
__global__ void dropout_scale_kernel(const float* __restrict__ in, const float* __restrict__ aux,
                                     OutT* __restrict__ out, int64_t n,
                                     uint32_t thr, float inv_keep, uint64_t seed,
                                     const uint64_t* __restrict__ seed_dev, uint32_t site) {
  pdl_grid_sync();
  if (thr && seed_dev) seed += *seed_dev;
  const int64_t nq = (n + 3) >> 2;
  for (int64_t q = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; q < nq;
       q += (int64_t)gridDim.x * blockDim.x) {
    const int64_t i0 = q << 2;
    u32x4 r = u32x4{~0u, ~0u, ~0u, ~0u};
    if (thr) r = dropout_bits4(seed, site, (uint64_t)q);
    if (i0 + 3 < n) {
      const float4 v = *reinterpret_cast<const float4*>(in + i0);
      float o[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
      for (int j = 0; j < 4; ++j) o[j] = (pick4(r, j) >= thr) ? o[j] * inv_keep : 0.f;
      if (aux) {
        const float4 a = *reinterpret_cast<const float4*>(aux + i0);
        if (!(a.x > 0.f)) o[0] = 0.f;
        if (!(a.y > 0.f)) o[1] = 0.f;
        if (!(a.z > 0.f)) o[2] = 0.f;
        if (!(a.w > 0.f)) o[3] = 0.f;
      }
#pragma unroll
      for (int j = 0; j < 4; ++j) out[i0 + j] = from_f32<OutT>(o[j]);
    } else {
      for (int j = 0; j < 4 && i0 + j < n; ++j)
        out[i0 + j] = from_f32<OutT>(((pick4(r, j) >= thr) && (!aux || aux[i0 + j] > 0.f)) ? in[i0 + j] * inv_keep : 0.f);
    }
  }
}

// ---------------------------------------------------------------------------
// embedding
// ---------------------------------------------------------------------------
__global__ void embed_fwd_kernel(const int64_t* __restrict__ idx, const float* __restrict__ tok,
                                 const float* __restrict__ pos, float* __restrict__ x, int M, int T,
                                 int C, int pos_offset) {
  pdl_grid_sync();
  // one warp per row (grid-stride); float4 when the row pitch allows it
  const int lane = threadIdx.x & 31;
  const int nwarp = (gridDim.x * blockDim.x) >> 5;
  const bool vec = (C & 3) == 0 && (((uintptr_t)tok | (uintptr_t)pos | (uintptr_t)x) & 15) == 0;
  for (int m = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; m < M; m += nwarp) {
    const float* tr = tok + idx[m] * (int64_t)C;
    const float* pr = pos ? pos + (int64_t)(m % T + pos_offset) * C : nullptr;
    float* xr = x + (int64_t)m * C;
    if (vec) {
      for (int q = lane; q < (C >> 2); q += 32) {
        float4 v = reinterpret_cast<const float4*>(tr)[q];
        if (pr) {
          const float4 w = reinterpret_cast<const float4*>(pr)[q];
          v.x += w.x; v.y += w.y; v.z += w.z; v.w += w.w;
        }
        reinterpret_cast<float4*>(xr)[q] = v;
      }
    } else {
      for (int c = lane; c < C; c += 32) xr[c] = tr[c] + (pr ? pr[c] : 0.f);
    }
  }
}

// dpos[t,c] += sum_b dx[b,t,c]  (deterministic: fixed summation order over b)
__global__ void embed_bwd_pos_kernel(const float* __restrict__ dx, float* __restrict__ dpos, int B,
                                     int T, int C, int pos_offset) {
  pdl_grid_sync();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= T * C) return;
  float acc = 0.f;
#pragma unroll 16
  for (int b = 0; b < B; ++b) acc += dx[(int64_t)b * T * C + i];  // independent loads: keep many in flight
  dpos[(int64_t)pos_offset * C + i] += acc;
}

// Fast token-gradient path when the whole [V, C] table fits in shared memory (80 x 384 fp32 = 120 KB):
// every CTA owns a slice of the rows and a private table; thread c adds dx[m, c] into table[idx[m]][c]
// (each thread touches only its own columns, so no atomics inside the CTA), then the rows of the
// table that were hit are added to the global gradient with one red.add per element.
__global__ void __launch_bounds__(512) embed_bwd_tok_smem_kernel(const int64_t* __restrict__ idx,
                                                                 const float* __restrict__ dx,
                                                                 float* __restrict__ dtok, int M, int C, int V,
                                                                 int rows_per_cta, int bulk) {
  pdl_grid_sync();
  extern __shared__ float table[];  // [V][C], hit flags [V], then this CTA's token ids [rows_per_cta]
  int* hit = reinterpret_cast<int*>(table + (size_t)V * C);
  int* ids = hit + V;
  const int r0 = blockIdx.x * rows_per_cta, r1 = min(M, r0 + rows_per_cta);
  for (int i = threadIdx.x; i < V * C; i += blockDim.x) table[i] = 0.f;
  for (int i = threadIdx.x; i < V; i += blockDim.x) hit[i] = 0;
  __syncthreads();
  for (int i = threadIdx.x; i < r1 - r0; i += blockDim.x) {  // ids up front: the row loop below is then one
    const int v = (int)idx[r0 + i];                           // stream of independent loads, 32 rows deep
    ids[i] = v;
    hit[v] = 1;
  }
  __syncthreads();
  constexpr int U = 32;  // rows in flight per thread: 128 B per thread, ~48 KB per SM (8 rows ran at 0.9 TB/s)
  for (int m = r0; m < r1; m += U) {
    for (int c = threadIdx.x; c < C; c += blockDim.x) {
      float x[U];
#pragma unroll
      for (int u = 0; u < U; ++u) x[u] = m + u < r1 ? dx[(int64_t)(m + u) * C + c] : 0.f;
#pragma unroll
      for (int u = 0; u < U; ++u)
        if (m + u < r1) table[ids[m + u - r0] * C + c] += x[u];
    }
  }
  // flush.  16-byte aligned gradient table: ONE bulk reduction of the whole shared-memory table (rows that were not hit
  // hold zeros) through the TMA unit -- the element-wise red.add loop below issued V * C atomics per CTA (4.5 M at the
  // benchmark shape) and was most of this kernel's 21 us.
  if (bulk) {
    ptx::fence_proxy_async();  // this thread's table writes -> visible to the async proxy
    __syncthreads();
    if (threadIdx.x == 0) {
      ptx::bulk_reduce_add_f32(dtok, table, (uint32_t)(V * C * sizeof(float)));
      ptx::bulk_commit();
      ptx::bulk_wait<0>();
    }
    return;
  }
  __syncthreads();
  for (int v = 0; v < V; ++v) {
    if (!hit[v]) continue;
    for (int c = threadIdx.x; c < C; c += blockDim.x) atomicAdd(&dtok[(int64_t)v * C + c], table[v * C + c]);
  }
}

// dtok[v, :] += sum_{m: idx[m]==v} dx[m, :]; one CTA per (v, 512-column chunk).
// The 80-row table would serialise global atomics, so each CTA scans idx (256 entries per
// step), builds an ORDERED list of matching rows in shared memory (deterministic sum order)
// and reduces them itself, two columns per thread.
__global__ void __launch_bounds__(256) embed_bwd_tok_kernel(const int64_t* __restrict__ idx,
                                                            const float* __restrict__ dx,
                                                            float* __restrict__ dtok, int M, int C) {
  __shared__ int list[256];
  __shared__ int warp_cnt[8];
  const int v = blockIdx.x;
  const int c0 = blockIdx.y * 512 + threadIdx.x, c1 = c0 + 256;
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  float acc0 = 0.f, acc1 = 0.f;
  for (int base = 0; base < M; base += 256) {
    const int m = base + threadIdx.x;
    const bool hit = (m < M) && (idx[m] == (int64_t)v);
    const unsigned bal = __ballot_sync(0xffffffffu, hit);
    if (lane == 0) warp_cnt[w] = __popc(bal);
    __syncthreads();
    int off = 0, total = 0;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      if (i < w) off += warp_cnt[i];
      total += warp_cnt[i];
    }
    if (hit) list[off + __popc(bal & ((1u << lane) - 1u))] = m;
    __syncthreads();
    for (int j = 0; j < total; ++j) {
      const float* row = dx + (int64_t)list[j] * C;
      if (c0 < C) acc0 += row[c0];
      if (c1 < C) acc1 += row[c1];
    }
    __syncthreads();
  }
  if (c0 < C) dtok[(int64_t)v * C + c0] += acc0;
  if (c1 < C) dtok[(int64_t)v * C + c1] += acc1;
}

// ---------------------------------------------------------------------------
// LayerNorm forward: one warp per row, row kept in registers (C <= 32*4*kMaxV)
// ---------------------------------------------------------------------------
static constexpr int kMaxV = 8;  // float4 per lane -> C <= 1024 on the register path

template <typename OutT>
__global__ void __launch_bounds__(256) ln_fwd_kernel(const float* __restrict__ x,
                                                     const float* __restrict__ gamma,
                                                     const float* __restrict__ beta,
                                                     OutT* __restrict__ y, float* __restrict__ mean,
                                                     float* __restrict__ rstd, int M, int C,
                                                     float eps) {
  const int lane = threadIdx.x & 31;
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= M) return;
  const float* xr = x + (int64_t)row * C;
  OutT* yr = y + (int64_t)row * C;
  if (gamma == nullptr) {  // identity cast
    for (int c = lane; c < C; c += 32) yr[c] = from_f32<OutT>(xr[c]);
    return;
  }
  if ((C & 3) == 0 && C <= 128 * kMaxV) {
    const int nv = C >> 2;
    float4 r[kMaxV];
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < kMaxV; ++i) {
      const int q = lane + 32 * i;
      if (q < nv) {
        r[i] = reinterpret_cast<const float4*>(xr)[q];
        s += (r[i].x + r[i].y) + (r[i].z + r[i].w);
      }
    }
    const float mu = warp_sum(s) / (float)C;
    float ss = 0.f;
#pragma unroll
    for (int i = 0; i < kMaxV; ++i) {
      const int q = lane + 32 * i;
      if (q < nv) {
        const float a = r[i].x - mu, b = r[i].y - mu, c = r[i].z - mu, d = r[i].w - mu;
        ss += (a * a + b * b) + (c * c + d * d);
      }
    }
    const float rs = rsqrtf(warp_sum(ss) / (float)C + eps);
    if (lane == 0) {
      mean[row] = mu;
      rstd[row] = rs;
    }
#pragma unroll
    for (int i = 0; i < kMaxV; ++i) {
      const int q = lane + 32 * i;
      if (q < nv) {
        const float4 g = reinterpret_cast<const float4*>(gamma)[q];
        const float4 b = reinterpret_cast<const float4*>(beta)[q];
        const float o0 = (r[i].x - mu) * rs * g.x + b.x, o1 = (r[i].y - mu) * rs * g.y + b.y;
        const float o2 = (r[i].z - mu) * rs * g.z + b.z, o3 = (r[i].w - mu) * rs * g.w + b.w;
        if constexpr (sizeof(OutT) == 4) {
          reinterpret_cast<float4*>(yr)[q] = make_float4(o0, o1, o2, o3);
        } else {
          __nv_bfloat162 lo = __floats2bfloat162_rn(o0, o1), hi = __floats2bfloat162_rn(o2, o3);
          uint2 pk;
          pk.x = *reinterpret_cast<uint32_t*>(&lo);
          pk.y = *reinterpret_cast<uint32_t*>(&hi);
          reinterpret_cast<uint2*>(yr)[q] = pk;
        }
      }
    }
    return;
  }
  // generic path
  float s = 0.f;
  for (int c = lane; c < C; c += 32) s += xr[c];
  const float mu = warp_sum(s) / (float)C;
  float ss = 0.f;
  for (int c = lane; c < C; c += 32) {
    const float d = xr[c] - mu;
    ss += d * d;
  }
  const float rs = rsqrtf(warp_sum(ss) / (float)C + eps);
  if (lane == 0) {
    mean[row] = mu;
    rstd[row] = rs;
  }
  for (int c = lane; c < C; c += 32)
    yr[c] = from_f32<OutT>((xr[c] - mu) * rs * gamma[c] + beta[c]);
}

// Streaming variant for C = 128 * NV: every warp normalises R rows at a time -- all of their loads are issued
// before the first reduction, which is what a memory-bound kernel with a two-stage dependent reduction per row
// needs (one row per warp kept ~1.5 KB in flight per warp and ran at ~3 TB/s).  EMBED: the rows are not read
// from x but built as tok[idx[m]] + pos[m % T + pos_offset] (src/model.py:595-597) and also written to x, i.e.
// the embedding lookup is fused with the first block's LayerNorm.
template <typename OutT, int NV, int R, bool EMBED>
__global__ void __launch_bounds__(256) ln_fwd_rows_kernel(float* __restrict__ x, const float* __restrict__ gamma,
                                                          const float* __restrict__ beta, OutT* __restrict__ y,
                                                          float* __restrict__ mean, float* __restrict__ rstd, int M,
                                                          float eps, const int64_t* __restrict__ idx,
                                                          const float* __restrict__ tok, const float* __restrict__ pos,
                                                          int T, int pos_offset) {
  pdl_grid_sync();
  constexpr int C = 128 * NV;
  const int lane = threadIdx.x & 31;
  const int nwarp = (gridDim.x * blockDim.x) >> 5;
  float4 g[NV], b[NV];
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    g[i] = reinterpret_cast<const float4*>(gamma)[lane + 32 * i];
    b[i] = reinterpret_cast<const float4*>(beta)[lane + 32 * i];
  }
  for (int row0 = ((blockIdx.x * blockDim.x + threadIdx.x) >> 5) * R; row0 < M; row0 += nwarp * R) {
    float4 r[R][NV];
    if (EMBED) {
      int64_t v[R];
#pragma unroll
      for (int k = 0; k < R; ++k) v[k] = row0 + k < M ? idx[row0 + k] : 0;
#pragma unroll
      for (int k = 0; k < R; ++k) {
        const int m = row0 + k;
        const float4* tr = reinterpret_cast<const float4*>(tok + v[k] * (int64_t)C);
        const float4* pr = reinterpret_cast<const float4*>(pos + (int64_t)((m < M ? m : 0) % T + pos_offset) * C);
#pragma unroll
        for (int i = 0; i < NV; ++i) {
          const float4 a = tr[lane + 32 * i], p = pr[lane + 32 * i];
          r[k][i] = make_float4(a.x + p.x, a.y + p.y, a.z + p.z, a.w + p.w);
        }
      }
    } else {
#pragma unroll
      for (int k = 0; k < R; ++k) {
        const float4* xr = reinterpret_cast<const float4*>(x + (int64_t)(row0 + k < M ? row0 + k : row0) * C);
#pragma unroll
        for (int i = 0; i < NV; ++i) r[k][i] = xr[lane + 32 * i];
      }
    }
    float s[R];
#pragma unroll
    for (int k = 0; k < R; ++k) {
      s[k] = 0.f;
#pragma unroll
      for (int i = 0; i < NV; ++i) s[k] += (r[k][i].x + r[k][i].y) + (r[k][i].z + r[k][i].w);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
      for (int k = 0; k < R; ++k) s[k] += __shfl_xor_sync(0xffffffffu, s[k], o);
    }
    float ss[R];
#pragma unroll
    for (int k = 0; k < R; ++k) {
      s[k] *= 1.f / (float)C;
      ss[k] = 0.f;
#pragma unroll
      for (int i = 0; i < NV; ++i) {
        const float a = r[k][i].x - s[k], bb = r[k][i].y - s[k], c = r[k][i].z - s[k], d = r[k][i].w - s[k];
        ss[k] += (a * a + bb * bb) + (c * c + d * d);
      }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
      for (int k = 0; k < R; ++k) ss[k] += __shfl_xor_sync(0xffffffffu, ss[k], o);
    }
#pragma unroll
    for (int k = 0; k < R; ++k) {
      const int m = row0 + k;
      if (m >= M) break;
      const float mu = s[k], rs = rsqrtf(ss[k] * (1.f / (float)C) + eps);
      if (lane == 0) {
        mean[m] = mu;
        rstd[m] = rs;
      }
      OutT* yr = y + (int64_t)m * C;
#pragma unroll
      for (int i = 0; i < NV; ++i) {
        const int q = lane + 32 * i;
        if (EMBED) reinterpret_cast<float4*>(x + (int64_t)m * C)[q] = r[k][i];
        const float o0 = (r[k][i].x - mu) * rs * g[i].x + b[i].x, o1 = (r[k][i].y - mu) * rs * g[i].y + b[i].y;
        const float o2 = (r[k][i].z - mu) * rs * g[i].z + b[i].z, o3 = (r[k][i].w - mu) * rs * g[i].w + b[i].w;
        if constexpr (sizeof(OutT) == 4) {
          reinterpret_cast<float4*>(yr)[q] = make_float4(o0, o1, o2, o3);
        } else {
          __nv_bfloat162 lo = __floats2bfloat162_rn(o0, o1), hi = __floats2bfloat162_rn(o2, o3);
          uint2 pk;
          pk.x = *reinterpret_cast<uint32_t*>(&lo);
          pk.y = *reinterpret_cast<uint32_t*>(&hi);
          reinterpret_cast<uint2*>(yr)[q] = pk;
        }
      }
    }
  }
}

// ---------------------------------------------------------------------------
// LayerNorm backward: warp per row (grid-stride), dgamma/dbeta reduced per CTA
// in shared memory, one global atomic per column per CTA.
// ---------------------------------------------------------------------------
template <typename DyT, typename MT>
__global__ void __launch_bounds__(256) ln_bwd_kernel(
    const DyT* __restrict__ dy, const float* __restrict__ x, const float* __restrict__ gamma,
    const float* __restrict__ mean, const float* __restrict__ rstd, const float* __restrict__ dres,
    float* __restrict__ dx, float* __restrict__ dgamma, float* __restrict__ dbeta,
    MT* __restrict__ dxm, uint32_t thr, float inv_keep, uint64_t seed,
    const uint64_t* __restrict__ seed_dev, uint32_t site, int M, int C) {
  extern __shared__ float sm[];  // [2*C]: dgamma, dbeta partials
  if (thr && seed_dev) seed += *seed_dev;
  float* sg = sm;
  float* sb = sm + C;
  for (int c = threadIdx.x; c < 2 * C; c += blockDim.x) sm[c] = 0.f;
  __syncthreads();
  const int lane = threadIdx.x & 31, wpb = blockDim.x >> 5;
  for (int row = blockIdx.x * wpb + (threadIdx.x >> 5); row < M; row += gridDim.x * wpb) {
    const float mu = mean[row], rs = rstd[row];
    const DyT* dyr = dy + (int64_t)row * C;
    const float* xr = x + (int64_t)row * C;
    float s1 = 0.f, s2 = 0.f;
    for (int c = lane; c < C; c += 32) {
      const float d = to_f32(dyr[c]);
      const float xh = (xr[c] - mu) * rs;
      const float dxh = d * gamma[c];
      s1 += dxh;
      s2 += dxh * xh;
      atomicAdd(&sg[c], d * xh);
      atomicAdd(&sb[c], d);
    }
    s1 = warp_sum(s1) / (float)C;
    s2 = warp_sum(s2) / (float)C;
    for (int c = lane; c < C; c += 32) {
      const float xh = (xr[c] - mu) * rs;
      float v = rs * (to_f32(dyr[c]) * gamma[c] - s1 - xh * s2);
      const int64_t i = (int64_t)row * C + c;
      if (dres) v += dres[i];
      dx[i] = v;
      if (dxm) {
        const bool keep = thr == 0 || dropout_keep(seed, site, (uint64_t)i, thr);
        dxm[i] = from_f32<MT>(keep ? v * inv_keep : 0.f);
      }
    }
  }
  __syncthreads();
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    atomicAdd(&dgamma[c], sg[c]);
    atomicAdd(&dbeta[c], sb[c]);
  }
}

// Fast path (C % 4 == 0, C <= 128*NV): each lane owns NV float4 column groups for every row its
// warp visits, so dgamma / dbeta / colsum(dxm) accumulate in registers (no shared-memory atomics);
// one cross-warp reduction and one global atomic per column per CTA at the end.  The optional
// colsum(dxm) output is the bias gradient of the GEMM that consumes dxm in the backward pass.
__device__ __forceinline__ float4 ld4(const float* p) { return *reinterpret_cast<const float4*>(p); }
__device__ __forceinline__ float4 ld4(const __nv_bfloat16* p) {
  const uint2 u = *reinterpret_cast<const uint2*>(p);
  const float2 a = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&u.x));
  const float2 b = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&u.y));
  return make_float4(a.x, a.y, b.x, b.y);
}
__device__ __forceinline__ void st4(float* p, float4 v) { *reinterpret_cast<float4*>(p) = v; }
__device__ __forceinline__ void st4(__nv_bfloat16* p, float4 v) {
  __nv_bfloat162 lo = __floats2bfloat162_rn(v.x, v.y), hi = __floats2bfloat162_rn(v.z, v.w);
  uint2 u;
  u.x = *reinterpret_cast<uint32_t*>(&lo);
  u.y = *reinterpret_cast<uint32_t*>(&hi);
  *reinterpret_cast<uint2*>(p) = u;
}

template <int NV, typename DyT, typename MT>
__global__ void __launch_bounds__(256, 2) ln_bwd_fast_kernel(
    const DyT* __restrict__ dy, const float* __restrict__ x, const float* __restrict__ gamma,
    const float* __restrict__ mean, const float* __restrict__ rstd, const float* __restrict__ dres,
    float* __restrict__ dx, float* __restrict__ dgamma, float* __restrict__ dbeta, MT* __restrict__ dxm,
    float* __restrict__ dxm_colsum, uint32_t thr, float inv_keep, uint64_t seed,
    const uint64_t* __restrict__ seed_dev, uint32_t site, int M, int C) {
  extern __shared__ float sm[];  // [8][C]
  if (thr && seed_dev) seed += *seed_dev;
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int nv = C >> 2;
  float4 g[NV], ag[NV], ab[NV], am[NV];
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int q = lane + 32 * i;
    g[i] = q < nv ? ld4(gamma + 4 * q) : make_float4(0.f, 0.f, 0.f, 0.f);
    ag[i] = ab[i] = am[i] = make_float4(0.f, 0.f, 0.f, 0.f);
  }
  const float invC = 1.f / (float)C;
  for (int row = blockIdx.x * 8 + w; row < M; row += gridDim.x * 8) {
    const float mu = mean[row], rs = rstd[row];
    const int64_t ro = (int64_t)row * C;
    float4 d[NV], xh[NV], rr[NV];
    float s1 = 0.f, s2 = 0.f;
#pragma unroll
    for (int i = 0; i < NV; ++i) {  // all three input streams in flight together
      const int q = lane + 32 * i;
      if (q < nv) {
        d[i] = ld4(dy + ro + 4 * q);
        xh[i] = ld4(x + ro + 4 * q);
        rr[i] = dres ? ld4(dres + ro + 4 * q) : make_float4(0.f, 0.f, 0.f, 0.f);
      }
    }
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      const int q = lane + 32 * i;
      if (q < nv) {
        const float4 xv = xh[i];
        xh[i] = make_float4((xv.x - mu) * rs, (xv.y - mu) * rs, (xv.z - mu) * rs, (xv.w - mu) * rs);
        const float4 t = make_float4(d[i].x * g[i].x, d[i].y * g[i].y, d[i].z * g[i].z, d[i].w * g[i].w);
        s1 += (t.x + t.y) + (t.z + t.w);
        s2 += (t.x * xh[i].x + t.y * xh[i].y) + (t.z * xh[i].z + t.w * xh[i].w);
        ag[i].x += d[i].x * xh[i].x; ag[i].y += d[i].y * xh[i].y; ag[i].z += d[i].z * xh[i].z; ag[i].w += d[i].w * xh[i].w;
        ab[i].x += d[i].x; ab[i].y += d[i].y; ab[i].z += d[i].z; ab[i].w += d[i].w;
      }
    }
    s1 = warp_sum(s1) * invC;
    s2 = warp_sum(s2) * invC;
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      const int q = lane + 32 * i;
      if (q < nv) {
        float4 v = make_float4(rs * (d[i].x * g[i].x - s1 - xh[i].x * s2), rs * (d[i].y * g[i].y - s1 - xh[i].y * s2),
                               rs * (d[i].z * g[i].z - s1 - xh[i].z * s2), rs * (d[i].w * g[i].w - s1 - xh[i].w * s2));
        v.x += rr[i].x; v.y += rr[i].y; v.z += rr[i].z; v.w += rr[i].w;
        st4(dx + ro + 4 * q, v);
        if (dxm) {
          if (thr) {
            const u32x4 b = dropout_bits4(seed, site, (uint64_t)row * (uint64_t)nv + (uint64_t)q);
            v.x = b.x >= thr ? v.x * inv_keep : 0.f;
            v.y = b.y >= thr ? v.y * inv_keep : 0.f;
            v.z = b.z >= thr ? v.z * inv_keep : 0.f;
            v.w = b.w >= thr ? v.w * inv_keep : 0.f;
          }
          st4(dxm + ro + 4 * q, v);
          am[i].x += v.x; am[i].y += v.y; am[i].z += v.z; am[i].w += v.w;
        }
      }
    }
  }
  // cross-warp reduction of the three column accumulators, one at a time through sm[8][C]
#pragma unroll 1
  for (int which = 0; which < 3; ++which) {
    float* out = which == 0 ? dgamma : which == 1 ? dbeta : dxm_colsum;
    if (out == nullptr) continue;
    __syncthreads();
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      const int q = lane + 32 * i;
      if (q < nv) st4(sm + w * C + 4 * q, which == 0 ? ag[i] : which == 1 ? ab[i] : am[i]);
    }
    __syncthreads();
    for (int c = threadIdx.x; c < C; c += 256) {
      float s = 0.f;
#pragma unroll
      for (int k = 0; k < 8; ++k) s += sm[k * C + c];
      atomicAdd(&out[c], s);
    }
  }
}

// Streaming version of the same math for the training shapes: a producer thread keeps a 4-deep ring of
// 8-row blocks (dy, x, dres, mean, rstd) in flight with cp.async.bulk + mbarriers, eight consumer warps
// take one row each out of shared memory.  Bytes in flight no longer depend on occupancy / registers
// (the register version stalled at ~35 % of HBM bandwidth with 16 resident warps per SM); one CTA per SM.
static constexpr int kLnRows = 8;     // rows per stage = consumer warps
static constexpr int kLnStages = 4;

template <int NV, typename DyT, typename MT>
__global__ void __launch_bounds__(32 + 32 * kLnRows, 1) ln_bwd_stream_kernel(
    const DyT* __restrict__ dy, const float* __restrict__ x, const float* __restrict__ gamma,
    const float* __restrict__ mean, const float* __restrict__ rstd, const float* __restrict__ dres,
    float* __restrict__ dx, float* __restrict__ dgamma, float* __restrict__ dbeta, MT* __restrict__ dxm,
    float* __restrict__ dxm_colsum, uint32_t thr, float inv_keep, uint64_t seed,
    const uint64_t* __restrict__ seed_dev, uint32_t site, int M, int C) {
  extern __shared__ __align__(128) uint8_t lsm[];
  using namespace ptx;
  const int dy_row = C * (int)sizeof(DyT), f_row = C * 4;
  const int stage_bytes = kLnRows * (dy_row + 2 * f_row) + 2 * kLnRows * 4 + 64;  // + mean, rstd (padded)
  const int stage_stride = (stage_bytes + 127) & ~127;
  uint64_t* full = reinterpret_cast<uint64_t*>(lsm + (size_t)kLnStages * stage_stride);
  uint64_t* empty = full + kLnStages;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int s = 0; s < kLnStages; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], kLnRows);
    }
    fence_barrier_init();
  }
  __syncthreads();
  pdl_grid_sync();  // barriers are set up; global memory from here on
  const int nblocks = (M + kLnRows - 1) / kLnRows;
  if (warp == 0) {
    if (lane == 0) {
      int s = 0;
      uint32_t ph = 0;
      for (int blk = blockIdx.x; blk < nblocks; blk += gridDim.x) {
        const int r0 = blk * kLnRows;
        const int nr = min(kLnRows, M - r0);
        mbar_wait(&empty[s], ph ^ 1);
        uint8_t* st = lsm + (size_t)s * stage_stride;
        const uint32_t bytes = nr * (dy_row + f_row + (dres ? f_row : 0)) + 2 * kLnRows * 4;
        mbar_expect_tx(&full[s], bytes);
        bulk_load_1d(st, dy + (int64_t)r0 * C, nr * dy_row, &full[s]);
        bulk_load_1d(st + kLnRows * dy_row, x + (int64_t)r0 * C, nr * f_row, &full[s]);
        if (dres) bulk_load_1d(st + kLnRows * (dy_row + f_row), dres + (int64_t)r0 * C, nr * f_row, &full[s]);
        // mean / rstd: always a full 32-byte copy (the arrays are padded by the caller's allocation granularity;
        // rows >= M are never consumed)
        bulk_load_1d(st + kLnRows * (dy_row + 2 * f_row), mean + r0, kLnRows * 4, &full[s]);
        bulk_load_1d(st + kLnRows * (dy_row + 2 * f_row) + kLnRows * 4, rstd + r0, kLnRows * 4, &full[s]);
        if (++s == kLnStages) { s = 0; ph ^= 1; }
      }
    }
    return;
  }
  // ------------------------------- consumers --------------------------------
  if (thr && seed_dev) seed += *seed_dev;
  const int cw = warp - 1;  // row inside the block
  const int nv = C >> 2;
  float4 g[NV], ag[NV], ab[NV], am[NV];
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int q = lane + 32 * i;
    g[i] = q < nv ? ld4(gamma + 4 * q) : make_float4(0.f, 0.f, 0.f, 0.f);
    ag[i] = ab[i] = am[i] = make_float4(0.f, 0.f, 0.f, 0.f);
  }
  const float invC = 1.f / (float)C;
  // Dropout mask of the bf16 copy.  With C % 32 == 0 a lane's float4 (quad q = lane + 32 i of the row) is always quad
  // (lane & 7) of its 32-element mask group, so the per-element multiplier / offset of the mask generator are four
  // per-thread constants (computed at run time they cost ~12 instructions per element), and the eight lanes that share
  // a group take its hash from the first of them instead of hashing eight times.
  const bool drop_fast = thr != 0;  // (the host only picks this kernel with dropout when C % 32 == 0)
  uint32_t dmul[4], dadd[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    dmul[k] = drop_mul((uint32_t)(lane & 7) * 4u + (uint32_t)k);
    dadd[k] = drop_add((uint32_t)(lane & 7) * 4u + (uint32_t)k);
  }
  int s = 0;
  uint32_t ph = 0;
  for (int blk = blockIdx.x; blk < nblocks; blk += gridDim.x) {
    const int row = blk * kLnRows + cw;
    mbar_wait(&full[s], ph);
    const uint8_t* st = lsm + (size_t)s * stage_stride;
    if (row < M) {
      const DyT* sdy = reinterpret_cast<const DyT*>(st) + cw * C;
      const float* sx = reinterpret_cast<const float*>(st + kLnRows * dy_row) + cw * C;
      const float* sr = reinterpret_cast<const float*>(st + kLnRows * (dy_row + f_row)) + cw * C;
      const float* sms = reinterpret_cast<const float*>(st + kLnRows * (dy_row + 2 * f_row));
      const float mu = sms[cw], rs = sms[kLnRows + cw];
      const int64_t ro = (int64_t)row * C;
      float4 d[NV], xh[NV];
      float s1 = 0.f, s2 = 0.f;
#pragma unroll
      for (int i = 0; i < NV; ++i) {
        const int q = lane + 32 * i;
        if (q < nv) {
          d[i] = ld4(sdy + 4 * q);
          const float4 xv = ld4(sx + 4 * q);
          xh[i] = make_float4((xv.x - mu) * rs, (xv.y - mu) * rs, (xv.z - mu) * rs, (xv.w - mu) * rs);
          const float4 t = make_float4(d[i].x * g[i].x, d[i].y * g[i].y, d[i].z * g[i].z, d[i].w * g[i].w);
          s1 += (t.x + t.y) + (t.z + t.w);
          s2 += (t.x * xh[i].x + t.y * xh[i].y) + (t.z * xh[i].z + t.w * xh[i].w);
          ag[i].x += d[i].x * xh[i].x; ag[i].y += d[i].y * xh[i].y; ag[i].z += d[i].z * xh[i].z; ag[i].w += d[i].w * xh[i].w;
          ab[i].x += d[i].x; ab[i].y += d[i].y; ab[i].z += d[i].z; ab[i].w += d[i].w;
        }
      }
      s1 = warp_sum(s1) * invC;
      s2 = warp_sum(s2) * invC;
#pragma unroll
      for (int i = 0; i < NV; ++i) {
        const int q = lane + 32 * i;
        if (q < nv) {
          float4 v = make_float4(rs * (d[i].x * g[i].x - s1 - xh[i].x * s2), rs * (d[i].y * g[i].y - s1 - xh[i].y * s2),
                                 rs * (d[i].z * g[i].z - s1 - xh[i].z * s2), rs * (d[i].w * g[i].w - s1 - xh[i].w * s2));
          if (dres) {
            const float4 r = ld4(sr + 4 * q);
            v.x += r.x; v.y += r.y; v.z += r.z; v.w += r.w;
          }
          st4(dx + ro + 4 * q, v);
          if (dxm) {
            if (drop_fast) {
              // (q < nv holds for all eight lanes of a group or for none: nv % 8 == 0, so the shuffles are safe)
              DropGroup dg = {0u, 0u};
              if ((lane & 7) == 0) dg = dropout_group(seed, site, ((uint64_t)row * (uint64_t)nv + (uint64_t)q) >> 3);
              const uint32_t h0 = __shfl_sync(0xffffffffu, dg.s0, lane & ~7), h1 = __shfl_sync(0xffffffffu, dg.s1, lane & ~7);
              v.x = h0 * dmul[0] + dadd[0] >= thr ? v.x * inv_keep : 0.f;
              v.y = h1 * dmul[1] + dadd[1] >= thr ? v.y * inv_keep : 0.f;
              v.z = h0 * dmul[2] + dadd[2] >= thr ? v.z * inv_keep : 0.f;
              v.w = h1 * dmul[3] + dadd[3] >= thr ? v.w * inv_keep : 0.f;
            }
            st4(dxm + ro + 4 * q, v);
            am[i].x += v.x; am[i].y += v.y; am[i].z += v.z; am[i].w += v.w;
          }
        }
      }
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(&empty[s]);
    if (++s == kLnStages) { s = 0; ph ^= 1; }
  }
  // cross-warp reduction of the three column accumulators through the (now idle) stage memory
  float* red = reinterpret_cast<float*>(lsm);
#pragma unroll 1
  for (int which = 0; which < 3; ++which) {
    float* out = which == 0 ? dgamma : which == 1 ? dbeta : dxm_colsum;
    if (out == nullptr) continue;
    asm volatile("bar.sync 1, 256;" ::: "memory");
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      const int q = lane + 32 * i;
      if (q < nv) st4(red + cw * C + 4 * q, which == 0 ? ag[i] : which == 1 ? ab[i] : am[i]);
    }
    asm volatile("bar.sync 1, 256;" ::: "memory");
    for (int c = threadIdx.x - 32; c < C; c += 256) {
      float sacc = 0.f;
#pragma unroll
      for (int k = 0; k < kLnRows; ++k) sacc += red[k * C + c];
      atomicAdd(&out[c], sacc);
    }
  }
}

// ---------------------------------------------------------------------------
// cross-entropy forward + backward, warp per row
// ---------------------------------------------------------------------------
template <typename DlT>
__global__ void __launch_bounds__(256) cross_entropy_kernel(
    const float* __restrict__ logits, int ld, const int64_t* __restrict__ targets,
    float* __restrict__ loss_sum, DlT* __restrict__ dlogits, int ld_dl,
    const float* __restrict__ dloss, int M, int V) {
  pdl_grid_sync();
  __shared__ float part[8];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int row = blockIdx.x * (blockDim.x >> 5) + w;
  float row_loss = 0.f;
  if (row < M) {
    const float* lr = logits + (int64_t)row * ld;
    float mx = -INFINITY;
    for (int v = lane; v < V; v += 32) mx = fmaxf(mx, lr[v]);
    mx = warp_max(mx);
    float se = 0.f;
    for (int v = lane; v < V; v += 32) se += expf(lr[v] - mx);
    se = warp_sum(se);
    const int tgt = (int)targets[row];
    row_loss = (logf(se) + mx - lr[tgt]) / (float)M;
    if (dlogits) {
      const float scale = (dloss ? dloss[0] : 1.f) / (float)M;
      const float inv = 1.f / se;
      DlT* dr = dlogits + (int64_t)row * ld_dl;
      for (int v = lane; v < V; v += 32) {
        const float p = expf(lr[v] - mx) * inv;
        dr[v] = from_f32<DlT>((p - (v == tgt ? 1.f : 0.f)) * scale);
      }
    }
  }
  if (lane == 0) part[w] = row_loss;
  __syncthreads();
  if (threadIdx.x == 0) {
    float s = 0.f;
    for (int i = 0; i < (int)(blockDim.x >> 5); ++i) s += part[i];
    atomicAdd(loss_sum, s);
  }
}

// ---------------------------------------------------------------------------
// flat AdamW
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(256) adamw_kernel(float* __restrict__ p, float* __restrict__ g,
                                                    float* __restrict__ m, float* __restrict__ v,
                                                    __nv_bfloat16* __restrict__ shadow, int64_t n,
                                                    const float* __restrict__ hyper,
                                                    const int64_t* __restrict__ step, int zero_grad) {
  pdl_grid_sync();
  const float lr = hyper[0], b1 = hyper[1], b2 = hyper[2], eps = hyper[3], wd = hyper[4], gs = hyper[5];
  const double t = (double)(*step + 1);
  const float bc1 = (float)(1.0 - pow((double)b1, t)), bc2 = (float)(1.0 - pow((double)b2, t));
  const float step_size = lr / bc1, inv_sqrt_bc2 = rsqrtf(bc2), decay = 1.f - lr * wd;
  const int64_t nq = n >> 2;
  for (int64_t q = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; q < nq;
       q += (int64_t)gridDim.x * blockDim.x) {
    float4 pp = reinterpret_cast<float4*>(p)[q];
    const float4 gg = reinterpret_cast<const float4*>(g)[q];
    float4 mm = reinterpret_cast<float4*>(m)[q];
    float4 vv = reinterpret_cast<float4*>(v)[q];
    float* pa = &pp.x; const float* ga = &gg.x; float* ma = &mm.x; float* va = &vv.x;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float gj = ga[j] * gs;
      pa[j] *= decay;
      ma[j] = ma[j] + (gj - ma[j]) * (1.f - b1);
      va[j] = va[j] * b2 + gj * gj * (1.f - b2);
      pa[j] -= step_size * ma[j] / (sqrtf(va[j]) * inv_sqrt_bc2 + eps);
    }
    reinterpret_cast<float4*>(p)[q] = pp;
    reinterpret_cast<float4*>(m)[q] = mm;
    reinterpret_cast<float4*>(v)[q] = vv;
    if (zero_grad) reinterpret_cast<float4*>(g)[q] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (shadow) {
      __nv_bfloat162 lo = __floats2bfloat162_rn(pp.x, pp.y), hi = __floats2bfloat162_rn(pp.z, pp.w);
      uint2 pk;
      pk.x = *reinterpret_cast<uint32_t*>(&lo);
      pk.y = *reinterpret_cast<uint32_t*>(&hi);
      reinterpret_cast<uint2*>(shadow)[q] = pk;
    }
  }
  // tail (n % 4)
  const int64_t i = (nq << 2) + blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i < n) {
    const float gj = g[i] * gs;
    float pj = p[i] * decay;
    const float mj = m[i] + (gj - m[i]) * (1.f - b1);
    const float vj = v[i] * b2 + gj * gj * (1.f - b2);
    pj -= step_size * mj / (sqrtf(vj) * inv_sqrt_bc2 + eps);
    p[i] = pj; m[i] = mj; v[i] = vj;
    if (zero_grad) g[i] = 0.f;
    if (shadow) shadow[i] = __float2bfloat16_rn(pj);
  }
}

__global__ void counter_add_kernel(uint64_t* ctr, uint64_t delta) {
  pdl_grid_sync();
  *ctr += delta;
}

__global__ void cast_bf16_kernel(const float* __restrict__ in, __nv_bfloat16* __restrict__ out,
                                 int64_t n) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n;
       i += (int64_t)gridDim.x * blockDim.x)
    out[i] = __float2bfloat16_rn(in[i]);
}

// ---------------------------------------------------------------------------
// column sums (bias gradients): each warp reads whole 128/256-column row segments with 16-byte
// loads (coalesced), 8 warps stride the rows, shared-memory reduce, one atomic per column per CTA
// ---------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256) colsum_kernel(const T* __restrict__ X, int M, int N, int ldx,
                                                     float* __restrict__ out, int rows_per_cta) {
  constexpr int VEC = sizeof(T) == 4 ? 4 : 8;  // elements per 16-byte load
  __shared__ float red[8][32 * VEC + 1];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int c0 = blockIdx.x * 32 * VEC + lane * VEC;
  const int r0 = blockIdx.y * rows_per_cta;
  const int r1 = min(M, r0 + rows_per_cta);
  float acc[VEC];
#pragma unroll
  for (int j = 0; j < VEC; ++j) acc[j] = 0.f;
  const bool vec = (c0 + VEC <= N) && (ldx % VEC == 0) && (((uintptr_t)X & 15) == 0);
  for (int r = r0 + w; r < r1; r += 8) {
    const T* p = X + (int64_t)r * ldx + c0;
    if (vec) {
      if constexpr (sizeof(T) == 4) {
        const float4 v = *reinterpret_cast<const float4*>(p);
        acc[0] += v.x; acc[1] += v.y; acc[2] += v.z; acc[3] += v.w;
      } else {
        const uint4 u = *reinterpret_cast<const uint4*>(p);
        const uint32_t uw[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float2 f = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&uw[j]));
          acc[2 * j] += f.x; acc[2 * j + 1] += f.y;
        }
      }
    } else {
#pragma unroll
      for (int j = 0; j < VEC; ++j)
        if (c0 + j < N) acc[j] += to_f32(p[j]);
    }
  }
#pragma unroll
  for (int j = 0; j < VEC; ++j) red[w][lane * VEC + j] = acc[j];
  __syncthreads();
  for (int c = threadIdx.x; c < 32 * VEC; c += 256) {
    const int col = blockIdx.x * 32 * VEC + c;
    if (col < N) {
      float s = 0.f;
#pragma unroll
      for (int k = 0; k < 8; ++k) s += red[k][c];
      atomicAdd(&out[col], s);
    }
  }
}

// ---------------------------------------------------------------------------
// sampler: one warp per sequence (the rule is warp_sample_row, sample.cuh)
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(32) sample_kernel(const float* __restrict__ logits, int ld,
                                                    int64_t* __restrict__ seq, int64_t seq_ld, int pos,
                                                    int V, int greedy, uint64_t seed,
                                                    const uint64_t* __restrict__ seed_dev, uint32_t step,
                                                    const dgpt_sampling* __restrict__ sampling) {
  const dgpt_sampling s = sampling ? *sampling : default_sampling();
  if (seed_dev) seed += *seed_dev;
  const int b = blockIdx.x;
  const int choice = warp_sample_row(logits + (int64_t)b * ld, V, greedy != 0, s, (uint32_t)b, step, seed);
  if (threadIdx.x == 0) seq[(int64_t)b * seq_ld + pos] = (int64_t)choice;
}

}  // namespace dgpt

using namespace dgpt;

// streaming LayerNorm forward (optionally fused with the embedding lookup); false = shape / alignment not covered
template <bool EMBED>
static bool launch_ln_rows(float* x, const float* gamma, const float* beta, void* y, int y_dtype, float* mean, float* rstd,
                           int M, int C, float eps, const int64_t* idx, const float* tok, const float* pos, int T,
                           int pos_offset, cudaStream_t st) {
  auto al16 = [](const void* q) { return ((uintptr_t)q & 15) == 0; };
  if (C % 128 != 0 || C > 512 || !gamma || !al16(x) || !al16(gamma) || !al16(beta) || !al16(y)) return false;
  if (EMBED && (!al16(tok) || !al16(pos))) return false;
  constexpr int R = 4;
  const int grid = min(ceil_div(M, 8 * R), kSMs * 4);
#define LN_ROWS(NV_)                                                                                              \
  case NV_:                                                                                                       \
    if (y_dtype == DGPT_F32)                                                                                      \
      launch_pdl(ln_fwd_rows_kernel<float, NV_, R, EMBED>, dim3(grid), dim3(256), 0, st, x, gamma, beta, (float*)y, mean, rstd, M, eps, idx, \
                                                                     tok, pos, T, pos_offset);                   \
    else                                                                                                          \
      launch_pdl(ln_fwd_rows_kernel<__nv_bfloat16, NV_, R, EMBED>, dim3(grid), dim3(256), 0, st, x, gamma, beta, (__nv_bfloat16*)y, mean,    \
                                                                             rstd, M, eps, idx, tok, pos, T, pos_offset); \
    break;
  switch (C / 128) {
    LN_ROWS(1)
    LN_ROWS(2)
    LN_ROWS(3)
    LN_ROWS(4)
    default: return false;
  }
#undef LN_ROWS
  return true;
}


extern "C" {

int dgpt_dropout_scale(const float* in, const float* relu_aux, void* out, int out_dtype, int64_t n, float p,
                       uint64_t seed, const uint64_t* seed_dev, uint32_t site, void* stream) {
  DGPT_DEVICE_OR_RETURN();
  DGPT_REQUIRE(p >= 0.f && p < 1.f, "dropout_scale: p=%f out of [0,1)", p);
  if (n == 0) return DGPT_OK;
  const uint32_t thr = dropout_threshold(p);
  const float inv_keep = 1.f / (1.f - p);
  const int grid = (int)min((int64_t)kSMs * 8, (n / 4 + 255) / 256 + 1);
  cudaStream_t st = (cudaStream_t)stream;
  if (out_dtype == DGPT_F32)
    launch_pdl(dropout_scale_kernel<float>, dim3(grid), dim3(256), 0, st, in, relu_aux, (float*)out, n, thr, inv_keep, seed, seed_dev, site);
  else
    launch_pdl(dropout_scale_kernel<__nv_bfloat16>, dim3(grid), dim3(256), 0, st, in, relu_aux, (__nv_bfloat16*)out, n, thr, inv_keep, seed, seed_dev, site);
  return check_launch("dropout_scale");
}

int dgpt_cast_bf16(const float* in, void* out, int64_t n, void* stream) {
  DGPT_DEVICE_OR_RETURN();
  if (n == 0) return DGPT_OK;
  const int grid = (int)min((int64_t)kSMs * 8, (n + 255) / 256);
  cast_bf16_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(in, (__nv_bfloat16*)out, n);
  return check_launch("cast_bf16");
}

int dgpt_embed_fwd(const int64_t* idx, const float* tok, const float* pos, float* x, int B, int T,
                   int C, int V, int pos_offset, void* stream) {
  DGPT_DEVICE_OR_RETURN();
  DGPT_REQUIRE(B >= 0 && T >= 0 && C > 0 && V > 0, "embed_fwd: bad shape B=%d T=%d C=%d V=%d", B, T, C, V);
  const int64_t total = (int64_t)B * T * C;
  if (total == 0) return DGPT_OK;
  const int grid = (int)min((int64_t)kSMs * 8, ((int64_t)B * T + 7) / 8);
  launch_pdl(embed_fwd_kernel, dim3(grid), dim3(256), 0, (cudaStream_t)stream, idx, tok, pos, x, B * T, T, C, pos_offset);
  return check_launch("embed_fwd");
}

int dgpt_embed_bwd(const int64_t* idx, const float* dx, float* dtok, float* dpos, int B, int T, int C,
                   int V, int pos_offset, void* stream) {
  DGPT_DEVICE_OR_RETURN();
  if ((int64_t)B * T == 0) return DGPT_OK;
  cudaStream_t st = (cudaStream_t)stream;
  if (dpos) launch_pdl(embed_bwd_pos_kernel, dim3(ceil_div((int64_t)T * C, 256)), dim3(256), 0, st, dx, dpos, B, T, C, pos_offset);
  const int M_ = B * T;
  const int ctas_ = min(kSMs, ceil_div(M_, 32));
  const size_t table_bytes = ((size_t)V * C + V + ceil_div(M_, ctas_)) * sizeof(float);
  // small problems keep the scan kernel: its summation order is deterministic (the 200-step parity runs at the
  // shipped checkpoints' shape are chaotic enough to notice atomics reordering)
  if (table_bytes <= 200 * 1024 && (int64_t)B * T >= 4096) {
    static bool attr = false;
    if (!attr) {
      cudaFuncSetAttribute(embed_bwd_tok_smem_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
      attr = true;
    }
    const int M = B * T;
    const int ctas = min(kSMs, ceil_div(M, 32));
    const int rows_per_cta = ceil_div(M, ctas);
    const int bulk = (((uintptr_t)dtok & 15) == 0 && ((size_t)V * C * sizeof(float)) % 16 == 0) ? 1 : 0;
    launch_pdl(embed_bwd_tok_smem_kernel, dim3(ceil_div(M, rows_per_cta)), dim3(384), table_bytes, st, idx, dx, dtok, M, C, V, rows_per_cta, bulk);
  } else {
    dim3 grid(V, ceil_div(C, 512));
    embed_bwd_tok_kernel<<<grid, 256, 0, st>>>(idx, dx, dtok, B * T, C);
  }
  return check_launch("embed_bwd");
}

int dgpt_ln_fwd(const float* x, const float* gamma, const float* beta, void* y, int y_dtype,
                float* mean, float* rstd, int M, int C, float eps, void* stream) {
  DGPT_DEVICE_OR_RETURN();
  if (M == 0) return DGPT_OK;
  DGPT_REQUIRE(C > 0, "ln_fwd: C=%d", C);
  cudaStream_t st = (cudaStream_t)stream;
  if (M >= 1024 && launch_ln_rows<false>(const_cast<float*>(x), gamma, beta, y, y_dtype, mean, rstd, M, C, eps, nullptr,
                                         nullptr, nullptr, 1, 0, st))
    return check_launch("ln_fwd");
  const int grid = ceil_div(M, 8);
  if (y_dtype == DGPT_F32)
    ln_fwd_kernel<float><<<grid, 256, 0, st>>>(x, gamma, beta, (float*)y, mean, rstd, M, C, eps);
  else
    ln_fwd_kernel<__nv_bfloat16><<<grid, 256, 0, st>>>(x, gamma, beta, (__nv_bfloat16*)y, mean, rstd, M, C, eps);
  return check_launch("ln_fwd");
}

// x[b,t,:] = tok[idx[b,t]] + pos[t + pos_offset] and y = LayerNorm(x) in one pass (src/model.py:595-597 followed by
// the first block's ln1, src/model_component.py:505).  Falls back to the two separate kernels for shapes the
// streaming kernel does not cover.
int dgpt_embed_ln_fwd(const int64_t* idx, const float* tok, const float* pos, float* x, const float* gamma,
                      const float* beta, void* y, int y_dtype, float* mean, float* rstd, int B, int T, int C, int V,
                      int pos_offset, float eps, void* stream) {
  DGPT_DEVICE_OR_RETURN();
  DGPT_REQUIRE(B >= 0 && T >= 0 && C > 0 && V > 0 && pos && gamma && beta, "embed_ln_fwd: bad arguments");
  if ((int64_t)B * T == 0) return DGPT_OK;
  cudaStream_t st = (cudaStream_t)stream;
  if (launch_ln_rows<true>(x, gamma, beta, y, y_dtype, mean, rstd, B * T, C, eps, idx, tok, pos, T, pos_offset, st))
    return check_launch("embed_ln_fwd");
  int rc = dgpt_embed_fwd(idx, tok, pos, x, B, T, C, V, pos_offset, stream);
  if (rc) return rc;
  return dgpt_ln_fwd(x, gamma, beta, y, y_dtype, mean, rstd, B * T, C, eps, stream);
}

int dgpt_ln_bwd(const void* dy, int dy_dtype, const float* x, const float* gamma, const float* mean,
                const float* rstd, const float* dres, float* dx, float* dgamma, float* dbeta,
                void* dxm, int dxm_dtype, float* dxm_colsum, float p, uint64_t seed,
                const uint64_t* seed_dev, uint32_t site, int M, int C, void* stream) {
  DGPT_DEVICE_OR_RETURN();
  if (M == 0) return DGPT_OK;
  DGPT_REQUIRE(C > 0 && C <= 6000, "ln_bwd: C=%d unsupported", C);
  DGPT_REQUIRE(p >= 0.f && p < 1.f, "ln_bwd: p=%f", p);
  DGPT_REQUIRE(!dxm_colsum || dxm, "ln_bwd: dxm_colsum needs dxm");
  cudaStream_t st = (cudaStream_t)stream;
  const uint32_t thr = dropout_threshold(p);
  const float ik = 1.f / (1.f - p);
  auto al = [](const void* q, uintptr_t a) { return ((uintptr_t)q & (a - 1)) == 0; };
  const bool fast = (C % 4 == 0) && C <= 1024 && al(x, 16) && al(gamma, 16) && al(dx, 16) && (!dres || al(dres, 16)) &&
                    al(dy, dy_dtype == DGPT_F32 ? 16 : 8) && (!dxm || al(dxm, dxm_dtype == DGPT_F32 ? 16 : 8));
  const bool stream_ok = fast && M >= 1024 && (C * (dy_dtype == DGPT_F32 ? 4 : 2)) % 16 == 0 && al(mean, 16) &&
                         al(rstd, 16) && al(dy, 16) && M % kLnRows == 0 && (thr == 0 || !dxm || C % 32 == 0);
  if (stream_ok) {
    const int dyb = dy_dtype == DGPT_F32 ? 4 : 2;
    const int stage_bytes = kLnRows * (C * dyb + 2 * C * 4) + 2 * kLnRows * 4 + 64;
    const size_t smem = (size_t)kLnStages * ((stage_bytes + 127) & ~127) + 2 * kLnStages * 8 + 64;
    const int nv = ceil_div(C, 128);
    const int grid = min(ceil_div(M, kLnRows), kSMs);
#define LN_STREAM(NV, DyT, MT)                                                                                       \
  do {                                                                                                               \
    static bool attr = false;                                                                                        \
    if (!attr) {                                                                                                     \
      cudaFuncSetAttribute(ln_bwd_stream_kernel<NV, DyT, MT>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024); \
      attr = true;                                                                                                   \
    }                                                                                                                \
    launch_pdl(ln_bwd_stream_kernel<NV, DyT, MT>, dim3(grid), dim3(32 + 32 * kLnRows), smem, st,                    \
               (const DyT*)dy, x, gamma, mean, rstd, dres, dx, dgamma, dbeta, (MT*)dxm, dxm_colsum, thr, ik, seed, seed_dev, \
               site, M, C);                                                                                          \
  } while (0)
#define LN_STREAM_T(NV)                                                                \
  do {                                                                                 \
    if (dy_dtype == DGPT_F32 && dxm_dtype == DGPT_F32) LN_STREAM(NV, float, float);    \
    else if (dy_dtype == DGPT_F32) LN_STREAM(NV, float, __nv_bfloat16);                \
    else if (dxm_dtype == DGPT_F32) LN_STREAM(NV, __nv_bfloat16, float);               \
    else LN_STREAM(NV, __nv_bfloat16, __nv_bfloat16);                                  \
  } while (0)
    if (smem <= 200 * 1024) {
      if (nv <= 1) LN_STREAM_T(1);
      else if (nv == 2) LN_STREAM_T(2);
      else if (nv == 3) LN_STREAM_T(3);
      else if (nv == 4) LN_STREAM_T(4);
      else LN_STREAM_T(8);
      return check_launch("ln_bwd_stream");
    }
#undef LN_STREAM_T
#undef LN_STREAM
  }
  if (fast) {
    const int grid = min(ceil_div(M, 8), kSMs * 2);
    const size_t smem = 8 * (size_t)C * sizeof(float);
    const int nv = ceil_div(C, 128);
#define LN_FAST(NV, DyT, MT)                                                                                   \
  ln_bwd_fast_kernel<NV, DyT, MT><<<grid, 256, smem, st>>>((const DyT*)dy, x, gamma, mean, rstd, dres, dx, dgamma, \
                                                           dbeta, (MT*)dxm, dxm_colsum, thr, ik, seed, seed_dev, site, M, C)
#define LN_FAST_T(NV)                                                                \
  do {                                                                               \
    if (dy_dtype == DGPT_F32 && dxm_dtype == DGPT_F32) LN_FAST(NV, float, float);    \
    else if (dy_dtype == DGPT_F32) LN_FAST(NV, float, __nv_bfloat16);                \
    else if (dxm_dtype == DGPT_F32) LN_FAST(NV, __nv_bfloat16, float);               \
    else LN_FAST(NV, __nv_bfloat16, __nv_bfloat16);                                  \
  } while (0)
    if (nv <= 1) LN_FAST_T(1);
    else if (nv == 2) LN_FAST_T(2);
    else if (nv == 3) LN_FAST_T(3);
    else if (nv == 4) LN_FAST_T(4);
    else LN_FAST_T(8);
#undef LN_FAST_T
#undef LN_FAST
    return check_launch("ln_bwd_fast");
  }
  const int grid = min(ceil_div(M, 8), kSMs * 4);
  const size_t smem = 2 * (size_t)C * sizeof(float);
#define LN_BWD(DyT, MT)                                                                             \
  ln_bwd_kernel<DyT, MT><<<grid, 256, smem, st>>>((const DyT*)dy, x, gamma, mean, rstd, dres, dx,   \
                                                  dgamma, dbeta, (MT*)dxm, thr, ik, seed, seed_dev, site, M, C)
  if (dy_dtype == DGPT_F32 && dxm_dtype == DGPT_F32) LN_BWD(float, float);
  else if (dy_dtype == DGPT_F32) LN_BWD(float, __nv_bfloat16);
  else if (dxm_dtype == DGPT_F32) LN_BWD(__nv_bfloat16, float);
  else LN_BWD(__nv_bfloat16, __nv_bfloat16);
#undef LN_BWD
  int rc = check_launch("ln_bwd");
  if (rc == DGPT_OK && dxm_colsum) rc = dgpt_colsum(dxm, dxm_dtype, M, C, C, dxm_colsum, 1, stream);
  return rc;
}

int dgpt_cross_entropy(const float* logits, int ld, const int64_t* targets, float* loss_sum,
                       void* dlogits, int dl_dtype, int ld_dl, const float* dloss, int M, int V,
                       void* stream) {
  DGPT_DEVICE_OR_RETURN();
  if (M == 0) return DGPT_OK;
  cudaStream_t st = (cudaStream_t)stream;
  const int grid = ceil_div(M, 8);
  if (dl_dtype == DGPT_F32)
    launch_pdl(cross_entropy_kernel<float>, dim3(grid), dim3(256), 0, st, logits, ld, targets, loss_sum, (float*)dlogits, ld_dl, dloss, M, V);
  else
    launch_pdl(cross_entropy_kernel<__nv_bfloat16>, dim3(grid), dim3(256), 0, st, logits, ld, targets, loss_sum, (__nv_bfloat16*)dlogits, ld_dl, dloss, M, V);
  return check_launch("cross_entropy");
}

int dgpt_counter_add(uint64_t* ctr, uint64_t delta, void* stream) {
  DGPT_DEVICE_OR_RETURN();
  launch_pdl(counter_add_kernel, dim3(1), dim3(1), 0, (cudaStream_t)stream, ctr, delta);
  return check_launch("counter_add");
}

int dgpt_adamw(float* p, float* g, float* m, float* v, void* shadow, int64_t n, const float* hyper,
               int64_t* step, int zero_grad, void* stream) {
  DGPT_DEVICE_OR_RETURN();
  if (n == 0) return DGPT_OK;
  DGPT_REQUIRE(hyper && step, "adamw: hyper/step must not be NULL");
  DGPT_REQUIRE((((uintptr_t)p | (uintptr_t)g | (uintptr_t)m | (uintptr_t)v) & 15) == 0 &&
                   (((uintptr_t)shadow) & 7) == 0,
               "adamw: arenas must be 16-byte aligned");
  const int grid = (int)min((int64_t)kSMs * 8, (n / 4 + 255) / 256 + 1);
  launch_pdl(adamw_kernel, dim3(grid), dim3(256), 0, (cudaStream_t)stream, p, g, m, v, (__nv_bfloat16*)shadow, n, hyper, step, zero_grad);
  launch_pdl(counter_add_kernel, dim3(1), dim3(1), 0, (cudaStream_t)stream, reinterpret_cast<uint64_t*>(step), 1ull);
  return check_launch("adamw");
}

int dgpt_colsum(const void* X, int dtype, int M, int N, int ldx, float* out, int accumulate,
                void* stream) {
  DGPT_DEVICE_OR_RETURN();
  if (N == 0) return DGPT_OK;
  cudaStream_t st = (cudaStream_t)stream;
  if (!accumulate) cudaMemsetAsync(out, 0, (size_t)N * sizeof(float), st);
  if (M == 0) return DGPT_OK;
  const int cols_per_cta = dtype == DGPT_F32 ? 128 : 256;
  const int gx = ceil_div(N, cols_per_cta);
  const int gy = max(1, min(ceil_div(M, 64), (kSMs * 4) / gx));
  const int rows_per_cta = ceil_div(M, gy);
  dim3 grid(gx, ceil_div(M, rows_per_cta));
  if (dtype == DGPT_F32)
    colsum_kernel<float><<<grid, 256, 0, st>>>((const float*)X, M, N, ldx, out, rows_per_cta);
  else
    colsum_kernel<__nv_bfloat16><<<grid, 256, 0, st>>>((const __nv_bfloat16*)X, M, N, ldx, out, rows_per_cta);
  return check_launch("colsum");
}

int dgpt_sample_ex(const float* logits, int ld, int64_t* seq, int64_t seq_ld, int pos, int B, int V,
                   int greedy, uint64_t seed, const uint64_t* seed_dev, uint32_t step,
                   const dgpt_sampling* sampling, void* stream) {
  DGPT_DEVICE_OR_RETURN();
  if (B == 0) return DGPT_OK;
  sample_kernel<<<B, 32, 0, (cudaStream_t)stream>>>(logits, ld, seq, seq_ld, pos, V, greedy, seed, seed_dev, step,
                                                    sampling);
  return check_launch("sample");
}

int dgpt_sample(const float* logits, int ld, int64_t* seq, int64_t seq_ld, int pos, int B, int V,
                int greedy, uint64_t seed, const uint64_t* seed_dev, uint32_t step, void* stream) {
  return dgpt_sample_ex(logits, ld, seq, seq_ld, pos, B, V, greedy, seed, seed_dev, step, nullptr, stream);
}

}  // extern "C"
