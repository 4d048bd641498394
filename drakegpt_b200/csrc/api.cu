// C-ABI dispatch for the GEMM and attention entry points: validates arguments and
// routes to the exact (fp32 CUDA-core) or tensor (bf16 tcgen05/TMA) kernels.
// Both are sm_100a CUDA; which one runs is decided by the operand dtype the
// caller passes, never by a runtime fallback.
#include "common.cuh"

namespace dgpt {
int launch_gemm_f32(const dgpt_gemm_args* a, cudaStream_t st);
int launch_gemm_tc(const dgpt_gemm_args* a, cudaStream_t st);
int launch_attn_fwd_simt(const dgpt_attn_args* a, cudaStream_t st);
int launch_attn_bwd_simt(const dgpt_attn_args* a, cudaStream_t st);
int launch_attn_fwd_tc(const dgpt_attn_args* a, cudaStream_t st);
int launch_attn_bwd_tc(const dgpt_attn_args* a, cudaStream_t st);
bool attn_tc_supported(const dgpt_attn_args* a);
}  // namespace dgpt

using namespace dgpt;

extern "C" {

int dgpt_gemm(const dgpt_gemm_args* a, void* stream) {
  DGPT_DEVICE_OR_RETURN();
  DGPT_REQUIRE(a != nullptr, "gemm: args is NULL");
  DGPT_REQUIRE(a->M >= 0 && a->N >= 0 && a->K >= 0, "gemm: negative shape M=%d N=%d K=%d", a->M, a->N, a->K);
  if (a->M == 0 || a->N == 0) return DGPT_OK;
  DGPT_REQUIRE(a->A && a->B && a->D, "gemm: A/B/D must not be NULL");
  DGPT_REQUIRE(a->dropout_p >= 0.f && a->dropout_p < 1.f, "gemm: dropout_p=%f", a->dropout_p);
  DGPT_REQUIRE(!a->accumulate || a->d_dtype == DGPT_F32, "gemm: accumulate needs an fp32 D");
  DGPT_REQUIRE(a->lda >= (a->a_major == DGPT_MAJOR_K ? a->K : a->M), "gemm: lda=%d too small", a->lda);
  DGPT_REQUIRE(a->ldb >= (a->b_major == DGPT_MAJOR_K ? a->K : a->N), "gemm: ldb=%d too small", a->ldb);
  DGPT_REQUIRE(a->ldd >= a->N, "gemm: ldd=%d < N=%d", a->ldd, a->N);
  if (a->split_k > 1)
    DGPT_REQUIRE(!a->relu && !a->relu_aux && a->dropout_p == 0.f && a->d_dtype == DGPT_F32 && !a->D2,
                 "gemm: split_k>1 only with a linear epilogue and fp32 D");
  cudaStream_t st = (cudaStream_t)stream;
  DGPT_REQUIRE(a->in_dtype == DGPT_BF16 || (!a->relu_mask_in && !a->relu_mask_out && !a->a_colsum),
               "gemm: relu_mask_in/out and a_colsum are tensor-mode (bf16) features");
  if (a->in_dtype == DGPT_F32) return launch_gemm_f32(a, st);
  if (a->in_dtype == DGPT_BF16) return launch_gemm_tc(a, st);
  set_error("gemm: unknown in_dtype %d", a->in_dtype);
  return DGPT_E_ARG;
}

static int check_attn(const dgpt_attn_args* a, const char* who) {
  DGPT_REQUIRE(a != nullptr, "%s: args is NULL", who);
  DGPT_REQUIRE(a->B >= 0 && a->NH > 0 && a->H > 0 && a->Tq >= 0 && a->Tk >= a->Tq,
               "%s: bad shape B=%d NH=%d H=%d Tq=%d Tk=%d", who, a->B, a->NH, a->H, a->Tq, a->Tk);
  DGPT_REQUIRE(a->dropout_p >= 0.f && a->dropout_p < 1.f, "%s: dropout_p=%f", who, a->dropout_p);
  DGPT_REQUIRE(a->dtype == DGPT_F32 || a->dtype == DGPT_BF16, "%s: dtype %d", who, a->dtype);
  return DGPT_OK;
}

int dgpt_attn_fwd(const dgpt_attn_args* a, void* stream) {
  DGPT_DEVICE_OR_RETURN();
  int rc = check_attn(a, "attn_fwd");
  if (rc) return rc;
  if (a->B == 0 || a->Tq == 0) return DGPT_OK;
  if (a->dtype == DGPT_BF16 && attn_tc_supported(a)) return launch_attn_fwd_tc(a, (cudaStream_t)stream);
  return launch_attn_fwd_simt(a, (cudaStream_t)stream);
}

int dgpt_attn_bwd(const dgpt_attn_args* a, void* stream) {
  DGPT_DEVICE_OR_RETURN();
  int rc = check_attn(a, "attn_bwd");
  if (rc) return rc;
  if (a->B == 0 || a->Tq == 0) return DGPT_OK;
  if (a->dtype == DGPT_BF16 && attn_tc_supported(a)) return launch_attn_bwd_tc(a, (cudaStream_t)stream);
  return launch_attn_bwd_simt(a, (cudaStream_t)stream);
}

int64_t dgpt_attn_bwd_scratch_bytes(const dgpt_attn_args* a) {
  if (!a) return 0;
  if (a->dtype == DGPT_BF16 && attn_tc_supported(a)) return 16;
  return (int64_t)a->B * a->NH * a->Tq * a->Tk * 2 * (int64_t)sizeof(float) + 16;
}

}  // extern "C"
