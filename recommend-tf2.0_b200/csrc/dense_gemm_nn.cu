// rtf_dense_gemm_nn: one layout of the fp32-accurate tensor-core GEMM (see dense_gemm.cuh); a
// translation unit per layout so the CUTLASS instantiations compile in parallel.
#include "dense_gemm.cuh"

using G = rtf_gemm::FastF32Gemm<rtf_gemm::RowMajor, rtf_gemm::RowMajor, RTF_GEMM_BANDS>;

extern "C" int rtf_dense_gemm_nn_workspace(int M, int N, int K, int batch, size_t* bytes) {
  if (!bytes) return RTF_E_ARG;
  return G::workspace(M, N, K, batch, bytes);
}

extern "C" int rtf_dense_gemm_nn(const float* d_a, int64_t lda, int64_t stride_a, const float* d_b,
                                 int64_t ldb, int64_t stride_b, const float* d_bias, int relu,
                                 float* d_out, int64_t ldd, int64_t stride_d, int M, int N, int K,
                                 int batch, void* d_ws, size_t ws_bytes, void* stream) {
  return G::run(d_a, lda, stride_a, d_b, ldb, stride_b, d_bias, relu, d_out, ldd, stride_d, M, N, K,
                batch, d_ws, ws_bytes, (cudaStream_t)stream);
}

using GP = rtf_gemm::FastF32PlanesGemm<rtf_gemm::RowMajor, rtf_gemm::RowMajor, RTF_GEMM_BANDS>;

extern "C" int rtf_dense_gemm_nn_planes_workspace(int M, int N, int K, int batch, size_t* bytes) {
  if (!bytes) return RTF_E_ARG;
  return GP::workspace(M, N, K, batch, bytes);
}

extern "C" int rtf_dense_gemm_nn_planes(const uint16_t* d_a, int64_t lda, int64_t stride_a,
                                        int64_t plane_a, const uint16_t* d_b, int64_t ldb,
                                        int64_t stride_b, int64_t plane_b, const float* d_bias,
                                        int relu, float* d_out, int64_t ldd, int64_t stride_d, int M,
                                        int N, int K, int batch, void* d_ws, size_t ws_bytes,
                                        void* stream) {
  return GP::run(d_a, lda, stride_a, plane_a, d_b, ldb, stride_b, plane_b, d_bias, relu, d_out, ldd,
                 stride_d, M, N, K, batch, d_ws, ws_bytes, (cudaStream_t)stream);
}
