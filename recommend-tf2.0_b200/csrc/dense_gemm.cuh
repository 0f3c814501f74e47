// Dense-MLP GEMMs (the MLP either side of the hot path, SURVEY.md §8 f2): fp32 in / fp32 out on
// the tcgen05 tensor cores with fp32-grade accuracy.
//
// Each fp32 operand is split on the fly into three bf16 terms x = x0 + x1 + x2 (8 + 8 + 8
// mantissa bits) and the product is accumulated from the bf16 partial products whose weight is
// >= 2^-16 of the leading one: x0*y0, x0*y1, x1*y0, x0*y2, x1*y1, x2*y0 ("3 bands", 6 UMMAs).
// The three products the library's BF16x9 emulation adds on top (x1*y2, x2*y1, x2*y2) weigh
// <= 2^-24 of the result, i.e. below one fp32 ulp, so they are skipped: 2/3 of the tensor work
// for the same fp32-level result (the parity bar is 1e-5; tests/test_dense_gemm_gpu.py measures
// ~1e-7 against fp64, the level of an IEEE fp32 GEMM).
//
// Configuration (tools/gemm_sweep, B200, M = 65 536): with the stock settings the kernel is bound by
// the accumulator promotion (TMEM -> registers after every K = 16 block), not by the MMAs: 5
// bands 141 vs 3 bands 154 TFLOP/s(fp32).  Promoting every 2 blocks (K = 32; measured error
// unchanged, 2.3e-7) and keeping the split A operand in shared memory instead of TMEM gives
// 201 TFLOP/s on the 1024x1024 layer vs 154 for cuBLAS 12.9's BF16x9 emulation; a source
// operand C (unused, beta = 0) costs 30 % through its shared-memory staging, so C is void.
//
// Built from the CUTLASS sm_100 collective for emulated fp32 (TMA loads -> transform warps split
// to bf16 into TMEM/shared memory -> tcgen05.mma with hardware accumulator scaling -> periodic
// promotion of the TMEM accumulator into fp32 registers -> fused bias + ReLU epilogue, TMA
// store), instantiated directly so that the band count is ours to choose (the stock builder
// fixes 5 bands = 9 products).  CUTLASS headers: the tree vendored in the image (see Makefile).
#pragma once
#include <cfloat>
#include <cstdint>
#include <cuda_runtime.h>

#include "cute/tensor.hpp"
#include "cutlass/cutlass.h"
#include "cutlass/epilogue/collective/collective_builder.hpp"
#include "cutlass/epilogue/fusion/operations.hpp"
#include "cutlass/epilogue/thread/activation.h"
#include "cutlass/gemm/collective/collective_builder.hpp"
#include "cutlass/gemm/device/gemm_universal_adapter.h"
#include "cutlass/gemm/kernel/gemm_universal.hpp"
#include "cutlass/numeric_types.h"

#include "rtf_b200.h"
#include "dense_gemm_planes.cuh"

namespace rtf_gemm {

using namespace cute;

using RowMajor = cutlass::layout::RowMajor;
using ColumnMajor = cutlass::layout::ColumnMajor;

// D[l] (M x N, row-major, ldd) = clamp(A[l] * B[l]^T + bias[n], lo, hi)
//   A[l]: logical (M x K); LayoutA RowMajor = K contiguous (lda between rows of M),
//                          ColumnMajor = M contiguous (lda between steps of K)
//   B[l]: logical (N x K); LayoutB ColumnMajor = K contiguous (ldb between rows of N),
//                          RowMajor = N contiguous (ldb between steps of K)
template <class LayoutA, class LayoutB, int Bands, class MmaTile = Shape<_256, _128, _32>,
          class Cluster = Shape<_2, _1, _1>,
          class MainSchedule = cutlass::gemm::KernelTmaWarpSpecialized2SmFastFP32SmemSm100,
          class EpiSchedule = cutlass::epilogue::TmaWarpSpecialized2Sm, class ElementC = void,
          int PromotionInterval = 2, class AccCopyAtom = void>
struct FastF32Gemm {
  using Arch = cutlass::arch::Sm100;
  using OpClass = cutlass::arch::OpClassTensorOp;
  using Fusion = cutlass::epilogue::fusion::LinCombPerColBiasEltAct<
      cutlass::epilogue::thread::Clamp, float, float, float, ElementC, float>;
  using Epilogue = typename cutlass::epilogue::collective::CollectiveBuilder<
      Arch, OpClass, MmaTile, Cluster, cutlass::epilogue::collective::EpilogueTileAuto, float,
      float, ElementC, RowMajor, 4, float, RowMajor, 4, EpiSchedule, Fusion>::CollectiveOp;
  using Stock = typename cutlass::gemm::collective::CollectiveBuilder<
      Arch, OpClass, float, LayoutA, 4, float, LayoutB, 4, float, MmaTile, Cluster,
      cutlass::gemm::collective::StageCountAutoCarveout<static_cast<int>(
          sizeof(typename Epilogue::SharedStorage))>,
      MainSchedule>::CollectiveOp;
  using SP = typename Stock::DispatchPolicy;
  using Policy = cutlass::gemm::MainloopSm100TmaUmmaWarpSpecializedFastF32<
      SP::Load2TransformPipelineStageCount, SP::Transform2MmaPipelineStageCount,
      SP::Schedule::SchedulerPipelineStageCount, SP::Schedule::AccumulatorPipelineStageCount, Bands,
      SP::ScalingFactor, (PromotionInterval > 0 ? PromotionInterval : SP::AccPromotionInterval),
      typename SP::ClusterShape,
      cute::conditional_t<cute::is_void_v<AccCopyAtom>, typename SP::AccumulatorCopyAtom, AccCopyAtom>,
      typename SP::ArchTag>;
  using Mainloop = cutlass::gemm::collective::CollectiveMma<
      Policy, typename Stock::TileShape, float, typename Stock::StrideA, float,
      typename Stock::StrideB, typename Stock::TiledMma, typename Stock::GmemTiledCopyA,
      typename Stock::SmemLayoutAtomsA, typename Stock::CopyAtomsA, typename Stock::TransformA,
      typename Stock::GmemTiledCopyB, typename Stock::SmemLayoutAtomsB, typename Stock::CopyAtomsB,
      typename Stock::TransformB>;
  using Kernel = cutlass::gemm::kernel::GemmUniversal<Shape<int, int, int, int>, Mainloop, Epilogue>;
  using Gemm = cutlass::gemm::device::GemmUniversalAdapter<Kernel>;
  using StrideA = typename Kernel::StrideA;
  using StrideB = typename Kernel::StrideB;
  using StrideD = typename Kernel::StrideD;

  // stride of a logical (rows x K [x batch]) operand: K contiguous -> (ld, 1, batch), else (1, ld, batch)
  template <class Stride, bool KContiguous>
  static Stride make_stride(int64_t ld, int64_t batch) {
    Stride s{};
    if constexpr (KContiguous) {
      get<0>(s) = ld;
    } else {
      get<1>(s) = ld;
    }
    get<2>(s) = batch;
    return s;
  }

  static typename Gemm::Arguments make_args(const float* A, int64_t lda, int64_t sA, const float* B,
                                            int64_t ldb, int64_t sB, const float* bias, float lo,
                                            float hi, float* D, int64_t ldd, int64_t sD, int M, int N,
                                            int K, int batch) {
    constexpr bool a_k = std::is_same_v<LayoutA, RowMajor>;
    constexpr bool b_k = std::is_same_v<LayoutB, ColumnMajor>;
    StrideA sa = make_stride<StrideA, a_k>(lda, sA);
    StrideB sb = make_stride<StrideB, b_k>(ldb, sB);
    StrideD sd = make_stride<StrideD, true>(ldd, sD);
    typename Gemm::Arguments args{cutlass::gemm::GemmUniversalMode::kGemm,
                                  {M, N, K, batch},
                                  {A, sa, B, sb},
                                  {{}, nullptr, sd, D, sd}};
    args.epilogue.thread.alpha = 1.f;
    args.epilogue.thread.beta = 0.f;
    args.epilogue.thread.bias_ptr = bias;
    args.epilogue.thread.activation.lower_bound = lo;
    args.epilogue.thread.activation.upper_bound = hi;
    static int sm_count = 0;
    int dev = 0;
    cudaGetDevice(&dev);
    if (sm_count == 0) cudaDeviceGetAttribute(&sm_count, cudaDevAttrMultiProcessorCount, dev);
    args.hw_info.device_id = dev;
    args.hw_info.sm_count = sm_count;
    return args;
  }

  static int workspace(int M, int N, int K, int batch, size_t* bytes) {
    auto args = make_args(nullptr, K, 0, nullptr, K, 0, nullptr, 0.f, 0.f, nullptr, N, 0, M, N, K, batch);
    *bytes = Gemm::get_workspace_size(args);
    return 0;
  }

  static int run(const float* A, int64_t lda, int64_t sA, const float* B, int64_t ldb, int64_t sB,
                 const float* bias, int relu, float* D, int64_t ldd, int64_t sD, int M, int N, int K,
                 int batch, void* ws, size_t ws_bytes, cudaStream_t st) {
    if (!A || !B || !D || M <= 0 || N <= 0 || K <= 0 || batch <= 0) return RTF_E_ARG;
    if (lda % 4 || ldb % 4 || ldd % 4 || sA % 4 || sB % 4 || sD % 4 || (uintptr_t)A % 16 ||
        (uintptr_t)B % 16 || (uintptr_t)D % 16 || (uintptr_t)bias % 16)
      return RTF_E_ALIGN;
    const float lo = relu ? 0.f : -INFINITY, hi = INFINITY;
    auto args = make_args(A, lda, sA, B, ldb, sB, bias, lo, hi, D, ldd, sD, M, N, K, batch);
    Gemm gemm;
    if (gemm.can_implement(args) != cutlass::Status::kSuccess) return RTF_E_RANGE;
    if (Gemm::get_workspace_size(args) > ws_bytes) return RTF_E_WORKSPACE;
    if (gemm.initialize(args, ws, st) != cutlass::Status::kSuccess) return RTF_E_ARG;
    cutlass::Status s = gemm.run(st);
    if (s != cutlass::Status::kSuccess) {
      const int e = (int)cudaGetLastError();  // read once: the call clears a non-sticky error
      return e ? e : RTF_E_ARG;
    }
    return 0;
  }
};

// The same GEMM fed pre-split bf16 planes (dense_gemm_planes.cuh): same tile, cluster, TiledMma
// (band order, ScalingFactor), promotion interval, accumulator stages and epilogue as
// FastF32Gemm, so D is bit-identical to FastF32Gemm's for the planes its transform would make.
// A[l] planes: bf16 at pa + p * pstride_a + <the fp32 operand's offset>, p = 0, 1, 2.
template <class LayoutA, class LayoutB, int Bands, int PromotionInterval = 2>
struct FastF32PlanesGemm {
  using Ref = FastF32Gemm<LayoutA, LayoutB, Bands>;
  using Epilogue = typename Ref::Epilogue;
  using SP = typename Ref::SP;
  using Stock = typename Ref::Stock;
  static constexpr bool a_k = std::is_same_v<LayoutA, RowMajor>;
  static constexpr bool b_k = std::is_same_v<LayoutB, ColumnMajor>;
  using StrideA = PlaneStride<a_k>;
  using StrideB = PlaneStride<b_k>;
  using TileShape = typename Stock::TileShape;
  using TiledMma = typename Stock::TiledMma;
  using AtomA = typename Stock::SmemLayoutAtomsA::ComputeLayoutAtom;
  using AtomB = typename Stock::SmemLayoutAtomsB::ComputeLayoutAtom;
  // bytes of one pipeline stage in one CTA: three bf16 planes of the A and B k-blocks
  static constexpr int kStageBytes =
      3 * 2 * (size<0>(TileShape{}) / 2 + size<1>(TileShape{}) / 2) * size<2>(TileShape{});
  static constexpr int kStages =
      (cutlass::arch::sm100_smem_capacity_bytes - static_cast<int>(sizeof(typename Epilogue::SharedStorage)) -
       4096) / kStageBytes;
  using Policy = MainloopSm100FastF32Planes<kStages, SP::Schedule::SchedulerPipelineStageCount,
                                            SP::Schedule::AccumulatorPipelineStageCount, Bands,
                                            SP::ScalingFactor, PromotionInterval, typename SP::ClusterShape>;
  using Mainloop = cutlass::gemm::collective::CollectiveMma<
      Policy, TileShape, cutlass::bfloat16_t, StrideA, cutlass::bfloat16_t, StrideB, TiledMma,
      cute::SM100_TMA_2SM_LOAD, AtomA, void, cute::identity, cute::SM100_TMA_2SM_LOAD, AtomB, void,
      cute::identity>;
  using Kernel = cutlass::gemm::kernel::GemmUniversal<Shape<int, int, int, int>, Mainloop, Epilogue>;
  using Gemm = cutlass::gemm::device::GemmUniversalAdapter<Kernel>;
  using StrideD = typename Kernel::StrideD;

  template <class Stride, bool KContiguous>
  static Stride make_stride(int64_t ld, int64_t batch, int64_t plane) {
    Stride s{};
    if constexpr (KContiguous) {
      get<0>(s) = ld;
    } else {
      get<1>(s) = ld;
    }
    get<2, 0>(s) = plane;
    get<2, 1>(s) = batch;
    return s;
  }

  static typename Gemm::Arguments make_args(const uint16_t* A, int64_t lda, int64_t sA, int64_t pA,
                                            const uint16_t* B, int64_t ldb, int64_t sB, int64_t pB,
                                            const float* bias, float lo, float hi, float* D,
                                            int64_t ldd, int64_t sD, int M, int N, int K, int batch) {
    StrideD sd = Ref::template make_stride<StrideD, true>(ldd, sD);
    typename Gemm::Arguments args{cutlass::gemm::GemmUniversalMode::kGemm,
                                  {M, N, K, batch},
                                  {reinterpret_cast<const cutlass::bfloat16_t*>(A),
                                   make_stride<StrideA, a_k>(lda, sA, pA),
                                   reinterpret_cast<const cutlass::bfloat16_t*>(B),
                                   make_stride<StrideB, b_k>(ldb, sB, pB)},
                                  {{}, nullptr, sd, D, sd}};
    args.epilogue.thread.alpha = 1.f;
    args.epilogue.thread.beta = 0.f;
    args.epilogue.thread.bias_ptr = bias;
    args.epilogue.thread.activation.lower_bound = lo;
    args.epilogue.thread.activation.upper_bound = hi;
    static int sm_count = 0;
    int dev = 0;
    cudaGetDevice(&dev);
    if (sm_count == 0) cudaDeviceGetAttribute(&sm_count, cudaDevAttrMultiProcessorCount, dev);
    args.hw_info.device_id = dev;
    args.hw_info.sm_count = sm_count;
    return args;
  }

  static int workspace(int M, int N, int K, int batch, size_t* bytes) {
    auto args = make_args(nullptr, K, 0, 0, nullptr, K, 0, 0, nullptr, 0.f, 0.f, nullptr, N, 0, M,
                          N, K, batch);
    *bytes = Gemm::get_workspace_size(args);
    return 0;
  }

  // bf16 TMA: 16-byte aligned bases and strides, i.e. every stride a multiple of 8 elements
  static int run(const uint16_t* A, int64_t lda, int64_t sA, int64_t pA, const uint16_t* B,
                 int64_t ldb, int64_t sB, int64_t pB, const float* bias, int relu, float* D,
                 int64_t ldd, int64_t sD, int M, int N, int K, int batch, void* ws, size_t ws_bytes,
                 cudaStream_t st) {
    if (!A || !B || !D || M <= 0 || N <= 0 || K <= 0 || batch <= 0 || pA <= 0 || pB <= 0)
      return RTF_E_ARG;
    if (lda % 8 || ldb % 8 || sA % 8 || sB % 8 || pA % 8 || pB % 8 || ldd % 4 || sD % 4 ||
        (uintptr_t)A % 16 || (uintptr_t)B % 16 || (uintptr_t)D % 16 || (uintptr_t)bias % 16)
      return RTF_E_ALIGN;
    const float lo = relu ? 0.f : -INFINITY, hi = INFINITY;
    auto args = make_args(A, lda, sA, pA, B, ldb, sB, pB, bias, lo, hi, D, ldd, sD, M, N, K, batch);
    Gemm gemm;
    if (gemm.can_implement(args) != cutlass::Status::kSuccess) return RTF_E_RANGE;
    if (Gemm::get_workspace_size(args) > ws_bytes) return RTF_E_WORKSPACE;
    if (gemm.initialize(args, ws, st) != cutlass::Status::kSuccess) return RTF_E_ARG;
    cutlass::Status s = gemm.run(st);
    if (s != cutlass::Status::kSuccess) {
      const int e = (int)cudaGetLastError();  // read once: the call clears a non-sticky error
      return e ? e : RTF_E_ARG;
    }
    return 0;
  }
};

}  // namespace rtf_gemm
