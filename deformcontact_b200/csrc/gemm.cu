// dc_gemm — C-ABI entry for the layer GEMMs; dispatches between the exact-fp32 SIMT kernel
// (gemm_simt.cu) and the tcgen05 3xTF32 tensor-core kernel (gemm_tc2.cu).
#include <stdlib.h>

#include "common.cuh"

namespace dcb {
size_t gemm_simt_workspace_bytes(int64_t M, int64_t N, int64_t Ktot);
int gemm_simt(const dc_gemm_seg* segs, int nseg, int transA, int transB, int64_t M, int64_t N, float* C, int64_t ldc,
              const float* bias, int relu, int accumulate, void* workspace, size_t workspace_bytes, cudaStream_t st);
bool gemm_tc2_supported(const dc_gemm_seg* segs, int nseg, int transA, int transB, int64_t M, int64_t N);
size_t gemm_tc2_workspace_bytes(int64_t M, int64_t N, int64_t Ktot);
int gemm_tc2(const dc_gemm_seg* segs, int nseg, int transA, int transB, int64_t M, int64_t N, float* C, int64_t ldc,
             const float* bias, int relu, int accumulate, void* workspace, size_t workspace_bytes, cudaStream_t st);
size_t gemm_tc2_batched_workspace_bytes(int count);
int gemm_tc2_batched(const dc_gemm_problem* probs, int count, int transA, int transB, int relu, int accumulate, void* workspace,
                     size_t workspace_bytes, void* host_staging, size_t host_staging_bytes, cudaStream_t st);
}  // namespace dcb

extern "C" size_t dc_gemm_batched_workspace_bytes(int32_t count) { return dcb::gemm_tc2_batched_workspace_bytes(count); }

extern "C" int dc_gemm_batched(const dc_gemm_problem* problems, int32_t count, int transA, int transB, int relu, int accumulate,
                               void* workspace, size_t workspace_bytes, void* host_staging, size_t host_staging_bytes,
                               dc_stream_t stream_) {
  DC_REQUIRE(count >= 0, DC_EINVAL, "gemm_batched: negative count");
  if (count == 0) return DC_OK;
  DC_REQUIRE(problems, DC_EINVAL, "gemm_batched: no problems");
  for (int32_t i = 0; i < count; ++i)
    DC_REQUIRE(!(problems[i].E && (relu || accumulate)), DC_EINVAL,
               "gemm_batched: problem %d: the fused epilogue operand E excludes relu and accumulate", i);
  return dcb::gemm_tc2_batched(problems, count, transA, transB, relu, accumulate, workspace, workspace_bytes, host_staging,
                               host_staging_bytes, (cudaStream_t)stream_);
}

extern "C" size_t dc_gemm_workspace_bytes(int64_t M, int64_t N, int64_t K_total, int transA, int transB) {
  (void)transA; (void)transB;
  if (M < 0 || N < 0 || K_total < 0) return 0;
  const size_t a = dcb::gemm_simt_workspace_bytes(M, N, K_total);
  const size_t b = dcb::gemm_tc2_workspace_bytes(M, N, K_total);
  return a > b ? a : b;
}

extern "C" int dc_gemm(const dc_gemm_seg* segs, int nseg, int transA, int transB, int64_t M, int64_t N, float* C,
                       int64_t ldc, const float* bias, int relu, int accumulate, int precision, void* workspace,
                       size_t workspace_bytes, dc_stream_t stream_) {
  cudaStream_t st = (cudaStream_t)stream_;
  DC_REQUIRE(segs && nseg >= 1 && nseg <= 4, DC_EINVAL, "gemm: nseg must be 1..4");
  DC_REQUIRE(M >= 0 && N >= 0, DC_EINVAL, "gemm: negative size");
  if (M == 0 || N == 0) return DC_OK;
  DC_REQUIRE(C && ldc >= N, DC_EINVAL, "gemm: bad C / ldc");
  DC_REQUIRE(precision >= DC_GEMM_AUTO && precision <= DC_GEMM_PREFER_TC, DC_EINVAL, "gemm: unknown precision %d", precision);
  if (precision != DC_GEMM_FP32) {
    const bool ok = dcb::gemm_tc2_supported(segs, nseg, transA, transB, M, N);
    if (precision == DC_GEMM_TF32X3) {
      DC_REQUIRE(ok, DC_ENOSUP, "gemm: shape/layout not supported by the tcgen05 path");
      return dcb::gemm_tc2(segs, nseg, transA, transB, M, N, C, ldc, bias, relu, accumulate, workspace, workspace_bytes, st);
    }
    // AUTO keeps small problems on the exact fp32 FFMA kernel; DCB200_DW_FP32=1 also keeps weight-gradient shaped
    // products (transposed A) there, as round 1 did (v1's long truncating accumulation chains cost accuracy; v2 cuts
    // every chain at 256 contraction elements and sums the chains in fp32 round-to-nearest)
    double work = (double)M * (double)N;
    int64_t ktot = 0;
    for (int s = 0; s < nseg; ++s) ktot += segs[s].K;
    work *= (double)ktot;
    static int dw_fp32 = -1;
    if (dw_fp32 < 0) { const char* e = getenv("DCB200_DW_FP32"); dw_fp32 = (e && e[0] == '1') ? 1 : 0; }
    if (ok && (precision == DC_GEMM_PREFER_TC || ((!transA || !dw_fp32) && work >= 1.0e8)))
      return dcb::gemm_tc2(segs, nseg, transA, transB, M, N, C, ldc, bias, relu, accumulate, workspace, workspace_bytes, st);
  }
  return dcb::gemm_simt(segs, nseg, transA, transB, M, N, C, ldc, bias, relu, accumulate, workspace, workspace_bytes, st);
}
