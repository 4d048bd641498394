/* drakegpt_b200 -- C-ABI of the hand-written sm_100a kernels behind the DrakeGPT
 * training step and generation path.
 *
 * The reference (ChrisTho23/DrakeGPT) has no FFI layer: its hot path is a chain
 * of PyTorch library calls.  Each entry point below replaces the group of
 * reference call sites cited next to it (file:line under the reference repo).
 * The host side (drakegpt_b200/*.py) binds these with ctypes and presents the
 * reference's own nn.Module API.
 *
 * Conventions
 *   - plain pointers and sizes only; every pointer is a DEVICE pointer unless
 *     the name ends in _host.  The caller owns all memory.
 *   - `stream` is a cudaStream_t passed as void*; kernels are enqueued on it and
 *     never synchronise or allocate, so every call is CUDA-graph capturable.
 *   - return 0 on success, a negative DGPT_E* code on failure;
 *     dgpt_last_error() returns a thread-local message for the last failure.
 *   - row-major tensors; "ld*" are leading dimensions in ELEMENTS.
 *   - dtype codes: DGPT_F32 = 0, DGPT_BF16 = 1.
 *   - no CPU fallback: every compute entry fails with DGPT_E_DEVICE when the
 *     current device is not compute capability 10.x.
 */
#ifndef DRAKEGPT_B200_H
#define DRAKEGPT_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DGPT_F32 0
#define DGPT_BF16 1

#define DGPT_OK 0
#define DGPT_E_ARG (-1)     /* bad shape / unsupported configuration            */
#define DGPT_E_DEVICE (-2)  /* no sm_100 device / driver entry point missing    */
#define DGPT_E_LAUNCH (-3)  /* cudaGetLastError() after the launch was non-zero */

#define DGPT_MAJOR_K 0  /* operand stored [rows, K], K contiguous                */
#define DGPT_MAJOR_MN 1 /* operand stored [K, rows], rows contiguous (transposed) */

const char* dgpt_last_error(void);
int dgpt_abi_version(void);
/* 0 when the current CUDA device is sm_100 and the TMA driver entry point resolves. */
int dgpt_device_check(void);
int dgpt_sm_count(void);
/* Diagnostics: with DGPT_CLOCK_PROBE=1 the GEMM and attention kernels stamp clock64 / %globaltimer in CTA 0;
 * returns the cycles and nanoseconds of the last stamped kernel (effective SM clock under load). Synchronises. */
int dgpt_debug_clock_probe(uint64_t* cycles, uint64_t* ns);
int dgpt_debug_clock_stamps(uint64_t* out64); /* raw stamps: [0..3] entry/exit clock64 + ns, [4..63] kernel phases */

/* ------------------------------------------------------------------------- *
 * Counter-based dropout mask shared by every kernel (forward and backward
 * regenerate it; nothing is stored).  Elements are taken in GROUPS of 32
 * consecutive indices; with g = i / 32, e = i % 32:
 *   h      = splitmix64(seed + g*0x9E3779B97F4A7C15 + (site+1)*0xD1B54A32D192ED03)
 *   s      = (e odd) ? high32(h) : low32(h)
 *   word   = s * MUL[e] + ADD[e]                      (mod 2^32; MUL[e] odd)
 *   keep(seed, site, i)  <=>  word >= round(p * 2^32)
 * MUL / ADD are the 32 per-position constants drop_mul(e) / drop_add(e) of
 * drakegpt_b200/csrc/common.cuh (integer finalisers of e): one 64-bit hash
 * per group, one 32-bit multiply-add per element.  The pairwise independence
 * of the 32 positions is tested in tests/test_cpu_host.py.
 * Replaces nn.Dropout at src/model_component.py:324,376/401,434/454.
 * Every entry that takes `seed` also takes `seed_dev`: an optional DEVICE
 * uint64 added to `seed` when the kernel runs, so that a captured CUDA graph
 * draws a fresh mask on every replay (the host bumps *seed_dev between
 * replays).  dgpt_dropout_keep_host is a host restatement used by the tests.
 * ------------------------------------------------------------------------- */
int dgpt_dropout_keep_host(uint64_t seed, uint32_t site, uint64_t index, float p);

/* out[i] = in[i] * keep(i) / (1-p) * (relu_aux ? relu_aux[i] > 0 : 1), cast to out_dtype
 * (p == 0 and relu_aux == NULL: plain cast).  relu_aux is fp32; it is the ReLU backward of
 * FeedForward (src/model_component.py:118-121). */
int dgpt_dropout_scale(const float* in, const float* relu_aux, void* out, int out_dtype, int64_t n,
                       float p, uint64_t seed, const uint64_t* seed_dev, uint32_t site,
                       void* stream);
/* fp32 -> bf16 copy (weight shadows for the tensor-core path). */
int dgpt_cast_bf16(const float* in, void* out, int64_t n, void* stream);

/* ------------------------------------------------------------------------- *
 * Embedding:  x[b,t,:] = tok[idx[b,t],:] (+ pos[t + pos_offset,:] if pos)
 * Replaces nn.Embedding x2 + add, src/model.py:595-597 (and :95 for BigramLM,
 * where pos == NULL and C == V).  idx is int64 like the reference's.
 * Backward: dtok[v,:] += sum_{idx==v} dx ; dpos[t+pos_offset,:] += sum_b dx.
 * ------------------------------------------------------------------------- */
int dgpt_embed_fwd(const int64_t* idx, const float* tok, const float* pos, float* x, int B, int T,
                   int C, int V, int pos_offset, void* stream);
int dgpt_embed_bwd(const int64_t* idx, const float* dx, float* dtok, float* dpos, int B, int T,
                   int C, int V, int pos_offset, void* stream);

/* ------------------------------------------------------------------------- *
 * LayerNorm (eps, biased variance, affine) -- nn.LayerNorm at
 * src/model_component.py:488-489, applied at :505-506.
 * fwd: y = (x-mean)*rstd*gamma+beta  cast to y_dtype; saves mean/rstd [M].
 *      gamma == NULL: y = cast(x) (identity; mean/rstd untouched).
 * bwd: dx = (dres ? dres : 0) + LN'(dy);  dgamma/dbeta are ACCUMULATED.
 *      Optional fused second output for the next backward GEMM:
 *      dxm = dx * keep(site)/(1-p) cast to dxm_dtype (dxm may be NULL), and
 *      dxm_colsum[c] += sum_m dxm[m,c] (may be NULL): the bias gradient of the
 *      Linear whose backward GEMMs consume dxm.
 * ------------------------------------------------------------------------- */
int dgpt_ln_fwd(const float* x, const float* gamma, const float* beta, void* y, int y_dtype,
                float* mean, float* rstd, int M, int C, float eps, void* stream);
/* Embedding lookup fused with the first block's LayerNorm: x[b,t,:] = tok[idx[b,t]] + pos[t + pos_offset]
 * (src/model.py:595-597) is written to x AND normalised into y in the same pass (ln1 of blocks.0,
 * src/model_component.py:505). */
int dgpt_embed_ln_fwd(const int64_t* idx, const float* tok, const float* pos, float* x, const float* gamma,
                      const float* beta, void* y, int y_dtype, float* mean, float* rstd, int B, int T, int C,
                      int V, int pos_offset, float eps, void* stream);
int dgpt_ln_bwd(const void* dy, int dy_dtype, const float* x, const float* gamma, const float* mean,
                const float* rstd, const float* dres, float* dx, float* dgamma, float* dbeta,
                void* dxm, int dxm_dtype, float* dxm_colsum, float p, uint64_t seed,
                const uint64_t* seed_dev, uint32_t site, int M, int C, void* stream);

/* ------------------------------------------------------------------------- *
 * GEMM with fused epilogue.   acc[m,n] = sum_k A(m,k) * B(n,k)
 *   A: a_major == K  -> stored [M,K] (lda >= K);  MN -> stored [K,M] (lda >= M)
 *   B: b_major == K  -> stored [N,K] (ldb >= K), i.e. an nn.Linear weight;
 *      MN -> stored [K,N] (ldb >= N)
 *   v = acc + bias[n]; relu; v *= (relu_aux[m,n] > 0); dropout(p,seed,site,
 *   index m*N+n); v += residual[m,n]; accumulate ? D += v : D = v;
 *   D (d_dtype) and optional D2 (d2_dtype) both receive v.
 * Replaces nn.Linear / `@` at src/model_component.py:392-393,404 (packed QKV),
 * :454 (proj + dropout + residual :505), :321-324 (FFN + ReLU + dropout +
 * residual :506), src/model.py:599 (lm_head) and their autograd backward
 * (dgrad: B MN-major; wgrad: A and B MN-major, split_k > 1 allowed).
 *   in_dtype DGPT_F32 : exact fp32 CUDA-core kernel, any shape.
 *   in_dtype DGPT_BF16: tcgen05/TMEM tiles fed by TMA, fp32 accumulate;
 *                       needs K % 8 == 0 and 16-byte aligned rows.
 * ------------------------------------------------------------------------- */
typedef struct dgpt_gemm_args {
  const void* A;
  const void* B;
  void* D;
  void* D2;               /* optional second output                         */
  const float* bias;      /* [N] or NULL                                    */
  const float* residual;  /* [M, ldr] fp32 or NULL                          */
  const void* relu_aux;   /* [M, ld_aux] (aux_dtype) or NULL                */
  int32_t M, N, K;
  int32_t in_dtype, d_dtype, d2_dtype, aux_dtype;
  int32_t a_major, b_major;
  int32_t lda, ldb, ldd, ldd2, ldr, ld_aux;
  int32_t relu;
  int32_t accumulate;     /* D += v (fp32 D only)                           */
  int32_t split_k;        /* >1: partial sums combined with fp32 atomics    */
  float dropout_p;
  uint32_t site;
  uint64_t seed;
  const uint64_t* seed_dev; /* optional device-side seed offset            */
  /* ReLU bit masks (tensor mode only; bf16 D, N % 64 == 0): word [(n / 32) * M + m] holds, in bit n % 32,
   * whether the pre-activation (m, n) was positive.  The forward GEMM (bias + relu) writes it, the dgrad
   * GEMM zeroes its output where the bit is clear -- 1/16 of the bytes of re-reading the bf16 activation
   * (src/model_component.py:321-322: Linear -> ReLU, and its autograd backward). */
  uint32_t* relu_mask_out;
  const uint32_t* relu_mask_in;
  /* Tensor mode, wgrad form (A and B MN-major, fp32 D): a_colsum[m] += sum_k A[m, k] -- with A = dY^T the bias
   * gradient of the Linear layer, computed on the tensor core inside the weight-gradient GEMM
   * (autograd of nn.Linear's bias, src/model_component.py:321-324). */
  float* a_colsum;
} dgpt_gemm_args;
int dgpt_gemm(const dgpt_gemm_args* a, void* stream);

/* out[n] (+)= sum_m X[m,n]   (bias gradients) */
int dgpt_colsum(const void* X, int dtype, int M, int N, int ldx, float* out, int accumulate,
                void* stream);

/* ------------------------------------------------------------------------- *
 * Fused causal attention over all heads.
 *   S = scale * Q K^T ; causal mask (query i sees keys j <= i + Tk - Tq);
 *   P = softmax(S) ; Pd = dropout(P) (no renormalisation) ; O = Pd V
 * Replaces, per head, src/model_component.py:56-64 / :396-405 and the concat
 * at :103/:260/:453 (head h is written at column h*H of O).
 *   q,k,v,o: element (b, t, h, d) at  base + b*bs + t*rs + h*H + d.
 *   lse[b,h,t] = log sum exp of the scaled, masked scores (saved for backward).
 *   dropout index = ((b*NH+h)*Tq + i)*Tk + j.
 *   dtype F32: exact CUDA-core kernel (any H<=128, Tk*H*8 bytes <= 200 KB).
 *   dtype BF16: tcgen05 kernel (H == 64, Tq == Tk, Tk % 128 == 0, Tk <= 256).
 * Backward needs `scratch` of dgpt_attn_bwd_scratch_bytes() bytes.
 * ------------------------------------------------------------------------- */
typedef struct dgpt_attn_args {
  const void* q;
  const void* k;
  const void* v;
  void* o;
  float* lse;
  const void* d_o; /* backward only */
  void* dq;
  void* dk;
  void* dv;
  void* scratch;
  int64_t q_bs, q_rs, k_bs, k_rs, v_bs, v_rs, o_bs, o_rs;
  int64_t dq_bs, dq_rs, dk_bs, dk_rs, dv_bs, dv_rs, do_bs, do_rs;
  int32_t dtype;
  int32_t B, NH, H, Tq, Tk;
  float scale;
  float dropout_p;
  uint32_t site;
  uint64_t seed;
  const uint64_t* seed_dev;
} dgpt_attn_args;
int dgpt_attn_fwd(const dgpt_attn_args* a, void* stream);
int dgpt_attn_bwd(const dgpt_attn_args* a, void* stream);
int64_t dgpt_attn_bwd_scratch_bytes(const dgpt_attn_args* a);

/* ------------------------------------------------------------------------- *
 * Cross-entropy over the character vocabulary, mean over rows.
 * Replaces F.cross_entropy at src/model.py:100-103,195-198,...,604-607.
 *   loss_sum[0] += sum_m (lse_m - logits[m,target_m]) / M      (pre-zeroed)
 *   dlogits[m,v] = (softmax(logits[m])[v] - [v==target_m]) * dloss / M
 * dlogits may be NULL (eval).  dloss is a device scalar or NULL (= 1).
 * ------------------------------------------------------------------------- */
int dgpt_cross_entropy(const float* logits, int ld, const int64_t* targets, float* loss_sum,
                       void* dlogits, int dl_dtype, int ld_dl, const float* dloss, int M, int V,
                       void* stream);

/* ------------------------------------------------------------------------- *
 * Fused LM head + cross-entropy (tensor mode): ONE kernel for
 *   logits = x . W^T + bias                     (src/model.py:599)
 *   loss   = F.cross_entropy(logits, targets)   (src/model.py:604-607)
 *   dlogits = (softmax(logits) - onehot(targets)) * dloss / M   (autograd)
 * x: bf16 [M, ldx] (K columns used); w: bf16 [V, ldw] (the nn.Linear weight).
 * One CTA per 128 rows: TMA -> tcgen05.mma 128 x V x 16 -> the logits row of
 * every token stays in TMEM, is reduced there (row max, sum of exponentials)
 * and only loss_sum[0] += sum_m (lse_m - logit[m, target_m]) / M (pre-zeroed
 * by the caller) and the bf16 dlogits [M, ld_dl] leave the chip.
 *   logits  (fp32 [M, ld_lg]) optional: written only when non-NULL (the API
 *           returns logits; the training step passes NULL).
 *   targets NULL: logits only (generation / eval without loss).
 *   dloss   device scalar or NULL (= 1).
 * Needs V % 16 == 0, 16 <= V <= 256, K % 64 == 0, K <= 512 and
 * K * (256 + 2 V) bytes <= 227 KB of shared memory (dgpt_lmhead_ce_supported);
 * other shapes use dgpt_gemm + dgpt_cross_entropy.
 * ------------------------------------------------------------------------- */
int dgpt_lmhead_ce_supported(int V, int K);
int dgpt_lmhead_ce(const void* x, int ldx, const void* w, int ldw, const float* bias,
                   const int64_t* targets, float* loss_sum, void* dlogits, int ld_dl,
                   float* logits, int ld_lg, const float* dloss, int M, int V, int K,
                   void* stream);

/* ------------------------------------------------------------------------- *
 * Residual GEMM with the next LayerNorm folded into its epilogue (tensor mode).
 * Replaces the tail of one transformer sub-block and the head of the next,
 * src/model_component.py:505-506 (x = x + sa(ln1(x)); x = x + ffwd(ln2(x))):
 *   x_out[M, N] (fp32) = dropout(a[M, K] @ w[N, K]^T + bias) + residual[M, N]
 *   y[M, N] (bf16) = (x_out - mean) * rstd * gamma + beta;  mean, rstd: [M]
 * a: bf16 [M, lda]; w: bf16 [N, ldw] (nn.Linear weight); residual / x_out:
 * fp32 with row pitches ldr / ldx; y: bf16 [M, ldy].  One CTA per 128 rows
 * holds the whole fp32 row in TMEM (tcgen05 128 x N x 16), so the statistics
 * need no second kernel and x_out makes no second trip through HBM.
 * Dropout (dropout_p > 0) uses the same counter-based mask as dgpt_gemm
 * (seed + *seed_dev, site, element index m * N + n), so dgpt_gemm's backward
 * twins regenerate it.  gamma == NULL: no normalisation, y is the bf16 copy of
 * x_out (the last block's output feeding the LM head); beta / mean / rstd unused.  Needs N in {128, 256, 384} and K % 64 == 0
 * (dgpt_gemm_res_ln_supported); other shapes use dgpt_gemm + dgpt_ln_fwd.
 * ------------------------------------------------------------------------- */
int dgpt_gemm_res_ln_supported(int N, int K);
int dgpt_gemm_res_ln(const void* a, int lda, const void* w, int ldw, const float* bias,
                     const float* residual, int ldr, float* x_out, int ldx,
                     const float* gamma, const float* beta, void* y, int ldy, float* mean,
                     float* rstd, int M, int N, int K, float eps, float dropout_p,
                     uint64_t seed, const uint64_t* seed_dev, uint32_t site, void* stream);

/* ------------------------------------------------------------------------- *
 * Fused flat AdamW (decoupled decay) over one parameter arena.
 * Replaces optimizer.zero_grad() + AdamW.step(), src/train.py:149,151
 * (torch.optim.AdamW defaults eps 1e-8, weight_decay 1e-2, SURVEY Q11).
 * hyper (device, 6 floats): lr, beta1, beta2, eps, weight_decay, grad_scale.
 * step (device int64): number of updates already applied; the kernel uses
 *   t = *step + 1 for the bias corrections and dgpt_adamw increments *step
 *   afterwards (on the stream), so a captured CUDA graph replays correctly
 *   without any host-side per-step state.
 *   g' = g*grad_scale; p *= 1-lr*wd; m = lerp(m,g',1-b1); v = b2*v+(1-b2)g'^2;
 *   p -= lr/(1-b1^t) * m / (sqrt(v)/sqrt(1-b2^t) + eps)
 * shadow (bf16, may be NULL) receives the updated weights; zero_grad != 0
 * clears g after use.
 * ------------------------------------------------------------------------- */
int dgpt_adamw(float* p, float* g, float* m, float* v, void* shadow, int64_t n,
               const float* hyper, int64_t* step, int zero_grad, void* stream);

/* ------------------------------------------------------------------------- *
 * Data-parallel optimizer step over NVLink peer memory (one process per GPU):
 * reduce-scatter of the gradient arenas + AdamW on this rank's 1/N shard +
 * all-gather of the updated fp32 parameters and bf16 shadows in ONE kernel
 * (P2P loads / stores on IPC-mapped peer arenas; two flag barriers).
 * Replaces the gradient mean a DDP wrapper would add around
 * src/train.py:149-151 plus optimizer.zero_grad() / AdamW.step(); the
 * reference itself is single-process (SURVEY 8e).
 *   dgpt_ipc_export / dgpt_ipc_open / dgpt_ipc_close: map a peer process's
 *     device buffer (handle = 64-byte cudaIpcMemHandle_t of the allocation,
 *     offset = position of the buffer inside it).
 *   peers: HOST array of 4*world + 1 device pointers -- g[world], p[world],
 *     shadow[world] (may be NULL), flags[world] (each 16 x uint32, zeroed
 *     once); entry [me] of each group is this rank's own buffer; the last
 *     entry is need32: one byte per 64-element block of the arena, non-zero
 *     where peers need the fp32 value (biases, LayerNorm, embeddings), zero for
 *     blocks that are only read through their bf16 shadows (GEMM weights: the
 *     fp32 master then stays with the owner), or NULL = broadcast everything.
 *   m, v: this rank's Adam moment shards ([hi - lo] floats); [lo, hi) is the
 *     64-element aligned shard of the arena this rank owns.
 *   hyper / step as dgpt_adamw (grad_scale = 1 / world for the mean);
 *   epoch (device uint32) and scratch (device 2 x uint32, zeroed once) are the
 *     barrier generation and {block counter, status}: status 1 / 2 = a peer
 *     never reached the first / second barrier within ~2 s (no hang).
 * The caller clears its gradient arena after this call (stream order).
 * ------------------------------------------------------------------------- */
int dgpt_ipc_export(const void* ptr, void* handle_out, int64_t* offset_out);
int dgpt_ipc_open(const void* handle, int64_t offset, void** ptr_out);
int dgpt_ipc_close(void* ptr, int64_t offset);
int dgpt_peer_copy(void* dst, const void* src, int64_t bytes, void* stream); /* one-sided fetch from a mapped peer buffer */
int dgpt_dp_adamw(const void* const* peers, int world, int me, float* m, float* v, int64_t lo,
                  int64_t hi, const float* hyper, int64_t* step, uint32_t* epoch,
                  uint32_t* scratch, int sms, void* stream);

/* *ctr += delta on the stream (dropout seed offsets under CUDA graphs). */
int dgpt_counter_add(uint64_t* ctr, uint64_t delta, void* stream);

/* ------------------------------------------------------------------------- *
 * Next-token sampling on the device.  Replaces
 * `logits[:, -1, :] -> F.softmax -> torch.multinomial -> torch.cat`,
 * src/model.py:628-635.  logits: row b at logits + b*ld ([V] fp32).
 *   greedy != 0: argmax (lowest index wins ties, like torch.argmax)
 *   else inverse-CDF sample with u = philox(seed + *seed_dev, step, b)  (seed_dev may be NULL).
 * Writes the token to seq[b*seq_ld + pos] (int64).
 *
 * dgpt_sample_ex also takes a DEVICE pointer to one dgpt_sampling struct;
 * NULL gives dgpt_sample's plain multinomial.  For one row l[0..V):
 *   1. top_k >= 1: keep v iff l[v] >= the k-th largest logit (ties kept);
 *      top_k <= 0 or >= V: off.
 *   2. e[v] = exp((l[v] - max) * (1 / temperature)) over the kept tokens,
 *      0 for the others.
 *   3. top_p < 1: order by e descending (lower index first on ties); keep v
 *      iff the sum of e over the tokens ahead of it is < top_p * sum(e).
 *   4. u = ((r.x >> 8) + 0.5) / 2^24 * (kept mass), r = philox4x32_10(b,
 *      step, 0x53414d50, 0; seed): the first v in vocabulary order whose
 *      inclusive cumulative kept mass is > u.
 * greedy ignores the settings (every filtered set contains the argmax).  With
 * temperature 1 and both cut-offs off the draw is exactly dgpt_sample's.  The
 * settings live in device memory so that one captured CUDA graph serves all.
 * The caller validates them (temperature > 0, 0 < top_p <= 1).
 * ------------------------------------------------------------------------- */
typedef struct dgpt_sampling {
  float temperature;
  int32_t top_k;
  float top_p;
} dgpt_sampling;
int dgpt_sample(const float* logits, int ld, int64_t* seq, int64_t seq_ld, int pos, int B, int V,
                int greedy, uint64_t seed, const uint64_t* seed_dev, uint32_t step, void* stream);
int dgpt_sample_ex(const float* logits, int ld, int64_t* seq, int64_t seq_ld, int pos, int B, int V,
                   int greedy, uint64_t seed, const uint64_t* seed_dev, uint32_t step,
                   const dgpt_sampling* sampling, void* stream);

/* ------------------------------------------------------------------------- *
 * KV-cached generation (tensor mode, head size 64, context <= 256) -- the
 * reference's generate loop, src/model.py:611-636, while the window has not slid.
 *
 * dgpt_decode_attn: ONE new query per (sequence, head) against nk cached
 *   keys / values (bf16): element (b, j, h, d) of k at k + b*k_bs + j*k_rs +
 *   h*64 + d (same for v); q / o: (b, h, d) at base + b*bs + h*64 + d.
 *   One warp per (b, h), lanes over keys, 16-byte loads: built to stream the
 *   KV cache at HBM speed for the large-batch end of the generation sweep.
 *
 * dgpt_decode_persistent: ONE launch for all positions t in [t0, t1) of up to
 *   dgpt_decode_persistent_max_batch() sequences: embedding, per layer
 *   LayerNorm + packed QKV matrix-vector product + KV append, attention,
 *   projection + residual, LayerNorm + FFN (+ReLU) + residual, then the LM head
 *   (ln_f is not applied, src/model.py:598-599) and the next token -- argmax
 *   (greedy != 0) or the same draw as dgpt_sample / dgpt_sample_ex
 *   (step = t) -- written to seq[(t+1)*B + b] for t >= t_sample.
 *   One thread-block CLUSTER (16 CTAs; `cluster` = 4 / 8 / 16, 0 = default) per
 *   group of <= 8 sequences, hardware cluster barriers between the phases, the
 *   weight rows of a phase prefetched into registers before the barrier it
 *   waits on; weights (bf16 shadows) stay L2-resident across tokens.
 *   layers: HOST array of nl x 12 device pointers per layer: wqkv [3D,C],
 *     wproj [C,D], w1 [F,C], w2 [C,F] (bf16), ln1 gamma/beta, ln2 gamma/beta,
 *     proj bias, b1, b2 (fp32), KV cache [B, ctx, 3D] (bf16, sequence-major).
 *   scratch: dgpt_decode_persistent_scratch_floats() floats.
 * dgpt_decode_persistent_supported: 1 if dgpt_decode_persistent takes this
 *   shape, else 0 (host only, needs no device).  The launch refuses exactly the
 *   shapes this refuses: head size 64, 1 <= B <= 8, 1 <= nl <= 8, C <= 512 and
 *   F <= 1536 (multiples of 8), NH * 64 <= 1536, ctx <= 256, cluster 4 / 8 / 16
 *   (<= 0: the size the launch would use), and every matrix-vector phase's
 *   rows (3D, F, V of K = C; C of K = D and of K = F) within the cluster's
 *   register budget: 12 rows per warp for K <= 512, 4 for K <= 1536.
 * ------------------------------------------------------------------------- */
int dgpt_decode_attn(const void* q, const void* k, const void* v, void* o, int64_t q_bs, int64_t k_bs,
                     int64_t k_rs, int64_t v_bs, int64_t v_rs, int64_t o_bs, int B, int NH, int H,
                     int nk, float scale, void* stream);
int64_t dgpt_decode_persistent_scratch_floats(int B, int C, int NH, int F, int V);
int dgpt_decode_persistent_max_batch(void);
int dgpt_decode_persistent_supported(int B, int nl, int C, int NH, int H, int F, int V, int ctx,
                                     int cluster);
int dgpt_decode_persistent(const void* const* layers, int nl, const float* tok, const float* pos,
                           const void* wlm, const float* blm, int64_t* seq, float* scratch, int B,
                           int C, int NH, int H, int F, int V, int ctx, int t0, int t1, int t_sample,
                           int greedy, uint64_t seed, const uint64_t* seed_dev, int cluster,
                           void* stream);
/* the same with the sampling settings of dgpt_sample_ex (device pointer, NULL = plain multinomial) */
int dgpt_decode_persistent_ex(const void* const* layers, int nl, const float* tok, const float* pos,
                              const void* wlm, const float* blm, int64_t* seq, float* scratch, int B,
                              int C, int NH, int H, int F, int V, int ctx, int t0, int t1,
                              int t_sample, int greedy, uint64_t seed, const uint64_t* seed_dev,
                              const dgpt_sampling* sampling, int cluster, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* DRAKEGPT_B200_H */
