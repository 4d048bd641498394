// Next-token rule shared by every decode path: dgpt_sample (sample_kernel) and the sampling phase of
// dgpt_decode_persistent.  One warp handles one row of fp32 logits l[0..V).
//
//   greedy: argmax, lowest index on ties (torch.argmax).  Otherwise, with the settings of dgpt_sampling:
//   1. top-k: v is kept iff l[v] >= the k-th largest logit (ties at the k-th value are kept); k <= 0 or k >= V: off
//   2. weight e[v] = exp((l[v] - max) * (1 / temperature)) for kept tokens, 0 for the others; S = sum of e
//   3. top-p: order the tokens by e descending, lower index first on ties; v stays kept iff the sum of e over the
//      tokens ahead of it is < top_p * S (the first token of that order always stays); top_p >= 1: off
//   4. draw: u = ((r.x >> 8) + 0.5) / 2^24 * S' with S' the kept mass and r = philox4x32_10(b, step, "SAMP", 0; seed);
//      the token is the first v in vocabulary order whose inclusive cumulative kept mass is > u
// With no settings (NULL), temperature 1 and both cut-offs off, the arithmetic is the plain softmax -> multinomial
// draw of the library's first sampler, operation for operation, so default streams do not change.
//
// The kept set after step 1 is {v : l[v] >= kth} and after step 3 a prefix of the (e desc, index asc) order, so both
// cut-offs reduce to one threshold each (kth; the last kept token (cut_e, cut_i)).  Ranks and "mass ahead" are counted
// over all V tokens per lane (O(V^2 / 32): V is a character vocabulary), with no per-lane arrays: every per-token
// value is recomputed from the logits row.  A run-time indexed array would go to local memory, which the persistent
// decoder cannot afford (its cluster barriers flush L1).
#pragma once
#include "common.cuh"

namespace dgpt {

// settings the caller loaded ahead of time (a device-memory load here would sit on the token's critical path)
__host__ __device__ __forceinline__ dgpt_sampling default_sampling() { return dgpt_sampling{1.f, 0, 1.f}; }

__device__ __forceinline__ int warp_sample_row(const float* lr, int V, bool greedy, const dgpt_sampling& sp, uint32_t b,
                                               uint32_t step, uint64_t seed) {
  const int lane = threadIdx.x & 31;
  float mx = -INFINITY;
  int arg = 0x7fffffff;
  for (int v = lane; v < V; v += 32) {
    const float l = lr[v];
    if (l > mx) { mx = l; arg = v; }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float om = __shfl_xor_sync(0xffffffffu, mx, o);
    const int oa = __shfl_xor_sync(0xffffffffu, arg, o);
    if (om > mx || (om == mx && oa < arg)) { mx = om; arg = oa; }
  }
  if (greedy) return arg;
  const float inv_t = sp.temperature == 1.f ? 1.f : 1.f / sp.temperature, top_p = sp.top_p;
  const int top_k = sp.top_k;
  const bool cut_k = top_k > 0 && top_k < V, cut_p = top_p < 1.f;
  // 1. top-k threshold: the smallest logit that fewer than k logits exceed
  float kth = -INFINITY;
  if (cut_k) {
    float lo = INFINITY;
    for (int v = lane; v < V; v += 32) {
      const float x = lr[v];
      int above = 0;
      for (int u = 0; u < V; ++u) above += lr[u] > x ? 1 : 0;
      if (above < top_k) lo = fminf(lo, x);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) lo = fminf(lo, __shfl_xor_sync(0xffffffffu, lo, o));
    kth = lo;
  }
  // 2. weights
  auto weight = [&](int v) {
    const float x = lr[v];
    return x >= kth ? expf((x - mx) * inv_t) : 0.f;
  };
  // 3. top-p: find the last token of the kept prefix
  float cut_e = 0.f;
  int cut_i = V;
  if (cut_p) {
    float s = 0.f;
    for (int v = lane; v < V; v += 32) s += weight(v);
    const float limit = top_p * warp_sum(s);
    float le = INFINITY;
    int li = -1;
    for (int v = lane; v < V; v += 32) {
      if (lr[v] < kth) continue;
      const float e = weight(v);
      float ahead = 0.f;
      for (int u = 0; u < V; ++u) {
        const float eu = weight(u);
        if (eu > e || (eu == e && u < v)) ahead += eu;
      }
      if ((ahead < limit || ahead == 0.f) && (e < le || (e == le && v > li))) { le = e; li = v; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float oe = __shfl_xor_sync(0xffffffffu, le, o);
      const int oi = __shfl_xor_sync(0xffffffffu, li, o);
      if (oe < le || (oe == le && oi > li)) { le = oe; li = oi; }
    }
    cut_e = le;
    cut_i = li;
  }
  // kept mass of token v (0 for a removed token)
  auto kept = [&](int v, float e) {
    return lr[v] >= kth && (!cut_p || e > cut_e || (e == cut_e && v <= cut_i));
  };
  // 4. inverse CDF over the kept mass in vocabulary order, 32 tokens per sweep
  float sk = 0.f;
  for (int v = lane; v < V; v += 32) {
    const float e = weight(v);
    if (kept(v, e)) sk += e;
  }
  sk = warp_sum(sk);
  const u32x4 r = philox4x32_10(b, step, 0x53414d50u /* "SAMP" */, 0u, (uint32_t)seed, (uint32_t)(seed >> 32));
  const float u = ((float)(r.x >> 8) + 0.5f) * (1.0f / 16777216.0f) * sk;  // target mass in (0, sk)
  float base = 0.f;
  int choice = -1, last = V - 1;  // last: the highest kept index, taken when rounding leaves u at the total
  for (int v0 = 0; v0 < V && choice < 0; v0 += 32) {
    const int v = v0 + lane;
    float e = 0.f;
    bool k = false;
    if (v < V) {
      e = weight(v);
      k = kept(v, e);
      if (!k) e = 0.f;
    }
    float c = e;  // inclusive scan
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const float t = __shfl_up_sync(0xffffffffu, c, o);
      if (lane >= o) c += t;
    }
    const unsigned hit = __ballot_sync(0xffffffffu, v < V && base + c > u);
    const unsigned kb = __ballot_sync(0xffffffffu, k);
    if (kb) last = v0 + 31 - __clz(kb);
    if (hit) choice = v0 + __ffs(hit) - 1;
    base += __shfl_sync(0xffffffffu, c, 31);
  }
  return choice >= 0 ? choice : last;
}

}  // namespace dgpt
