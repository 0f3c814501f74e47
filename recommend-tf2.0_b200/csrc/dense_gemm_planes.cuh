// Plane-fed mainloop for the dense-MLP GEMM (dense_gemm.cuh): the operands arrive already split
// into three bf16 planes x = x0 + x1 * 2^-S + x2 * 2^-2S (rtf::split_bf16x3, rtf_common.cuh), so
// the mainloop needs no transform warps.  The TMA producer loads the planes straight into the
// shared-memory buffers the MMA warp reads; the MMA warp issues the same 6 (3 bands) scaled UMMAs
// in the same order as CUTLASS's emulated FastF32 collective
// (cutlass/gemm/collective/sm100_mma_warpspecialized_emulated.hpp), and the epilogue warps promote
// the TMEM accumulator into fp32 registers with the same adds.  Fed the planes the fp32 mainloop
// would have made, the result is therefore bit-identical to the fp32-fed kernel.
//
// The collective plugs into CUTLASS's sm100 "MMA transform" kernel
// (sm100_gemm_tma_warpspecialized_mma_transform.hpp: load warp -> MMA warp -> epilogue warps that
// post-process the accumulator), the kernel the blockwise-scaled GEMMs use.  That kernel also
// runs a scale-factor load warp; here it has nothing to load and returns at once.
//
// Operand in global memory: one bf16 tensor (3, rows, ld) per operand, i.e. plane p of logical
// element (r, k[, l]) at p * plane_stride + <the fp32 operand's offset>.  The plane index rides on
// the batch mode, (M, K, (3, L)), so each k-block of a plane is one TMA box.
#pragma once
#include "cutlass/gemm/collective/collective_builder.hpp"
#include "cutlass/gemm/kernel/gemm_universal.hpp"

namespace rtf_gemm {

template <int Stages_, int SchedulerPipelineStageCount_, int AccumulatorPipelineStageCount_,
          int NumBandsToCompute_, int ScalingFactor_, int AccPromotionInterval_, class ClusterShape_>
struct MainloopSm100FastF32Planes {
  constexpr static int Stages = Stages_;
  constexpr static int NumBandsToCompute = NumBandsToCompute_;
  constexpr static int ScalingFactor = ScalingFactor_;
  constexpr static int AccPromotionInterval = AccPromotionInterval_;
  using ClusterShape = ClusterShape_;
  using ArchTag = cutlass::arch::Sm100;
  using Schedule = cutlass::gemm::KernelTmaWarpSpecializedMmaTransformSm100<
      SchedulerPipelineStageCount_, AccumulatorPipelineStageCount_>;
  constexpr static bool IsOverlappingAccum = false;
};

// stride of a plane operand: (rows, K, (plane, batch))
template <bool KContiguous>
using PlaneStride = cute::conditional_t<
    KContiguous, cute::Stride<int64_t, cute::_1, cute::Stride<int64_t, int64_t>>,
    cute::Stride<cute::_1, int64_t, cute::Stride<int64_t, int64_t>>>;

}  // namespace rtf_gemm

namespace cutlass::gemm::collective {
using namespace cute;

template <int Stages, int SchedulerPipelineStageCount, int AccumulatorPipelineStageCount_,
          int NumBandsToCompute_, int ScalingFactor_, int AccPromotionInterval_, class ClusterShape,
          class TileShape_, class StrideA_, class StrideB_, class TiledMma_, class SmemLayoutAtomA_,
          class SmemLayoutAtomB_>
struct CollectiveMma<
    rtf_gemm::MainloopSm100FastF32Planes<Stages, SchedulerPipelineStageCount,
                                         AccumulatorPipelineStageCount_, NumBandsToCompute_,
                                         ScalingFactor_, AccPromotionInterval_, ClusterShape>,
    TileShape_, cutlass::bfloat16_t, StrideA_, cutlass::bfloat16_t, StrideB_, TiledMma_,
    SM100_TMA_2SM_LOAD, SmemLayoutAtomA_, void, cute::identity, SM100_TMA_2SM_LOAD,
    SmemLayoutAtomB_, void, cute::identity> {
  using TiledMma = TiledMma_;
  using AtomThrShapeMNK = Shape<decltype(shape<0>(typename TiledMma::ThrLayoutVMNK{})), _1, _1>;
  using DispatchPolicy =
      rtf_gemm::MainloopSm100FastF32Planes<Stages, SchedulerPipelineStageCount,
                                           AccumulatorPipelineStageCount_, NumBandsToCompute_,
                                           ScalingFactor_, AccPromotionInterval_, ClusterShape>;
  using TileShape = TileShape_;
  using ElementA = cutlass::bfloat16_t;
  using ElementB = cutlass::bfloat16_t;
  using ElementAMma = typename TiledMma::ValTypeA;
  using ElementBMma = typename TiledMma::ValTypeB;
  using StrideA = StrideA_;
  using StrideB = StrideB_;
  using ElementAccumulator = typename TiledMma::ValTypeC;
  using GmemTiledCopyA = SM100_TMA_2SM_LOAD;
  using GmemTiledCopyB = SM100_TMA_2SM_LOAD;
  using SmemLayoutAtomA = SmemLayoutAtomA_;
  using SmemLayoutAtomB = SmemLayoutAtomB_;
  using SmemCopyAtomA = void;
  using SmemCopyAtomB = void;
  using TransformA = cute::identity;
  using TransformB = cute::identity;
  using ArchTag = typename DispatchPolicy::ArchTag;

  static_assert(cute::is_same_v<ElementAMma, cutlass::bfloat16_t> &&
                cute::is_same_v<ElementBMma, cutlass::bfloat16_t>);
  static_assert(size(AtomThrShapeMNK{}) == 2, "written for the 2-SM UMMA");
  static_assert(cute::is_static_v<ClusterShape>);
  static_assert(cute::is_base_of<cute::UMMA::DescriptorIterator, typename TiledMma::FrgTypeA>::value &&
                    cute::is_base_of<cute::UMMA::DescriptorIterator, typename TiledMma::FrgTypeB>::value,
                "both operands are read from shared memory");

  using CtaShape_MNK = decltype(shape_div(TileShape{}, AtomThrShapeMNK{}));
  using MmaShapeA_MK = decltype(partition_shape_A(
      TiledMma{}, make_shape(size<0>(TileShape{}), size<2>(TileShape{}))));
  using MmaShapeB_NK = decltype(partition_shape_B(
      TiledMma{}, make_shape(size<1>(TileShape{}), size<2>(TileShape{}))));

  constexpr static int NumComputeMtxs = 3;
  constexpr static int NumBandsToCompute = NumBandsToCompute_;
  constexpr static int ScalingFactor = ScalingFactor_;
  constexpr static int AccPromotionInterval = AccPromotionInterval_;
  constexpr static int AccumulatorPipelineStageCount = AccumulatorPipelineStageCount_;
  constexpr static int StagesPerTile = size<2>(MmaShapeA_MK{}) / AccPromotionInterval;
  static_assert(NumBandsToCompute >= 3 && NumBandsToCompute <= 5);
  static_assert(size<2>(MmaShapeA_MK{}) % AccPromotionInterval == 0);

  using MainloopABPipeline = cutlass::PipelineTmaUmmaAsync<Stages, ClusterShape, AtomThrShapeMNK>;
  using MainloopABPipelineState = typename MainloopABPipeline::PipelineState;
  // the kernel's scale-factor pipeline: allocated, never used
  using MainloopSFPipeline = cutlass::PipelineAsync<1>;
  using MainloopSFPipelineState = typename MainloopSFPipeline::PipelineState;
  using AccumulatorPipeline = cutlass::PipelineUmmaAsync<AccumulatorPipelineStageCount, AtomThrShapeMNK>;
  using AccumulatorPipelineState = typename AccumulatorPipeline::PipelineState;
  static constexpr int NumMainloopSFProducerThreadEvents = 1;

  // (MMA, MMA_M|N, MMA_K, PLANE + 3 * PIPE): the three planes of a stage sit side by side
  using SmemLayoutA = decltype(UMMA::tile_to_mma_shape(
      SmemLayoutAtomA{}, append(MmaShapeA_MK{}, Int<NumComputeMtxs * Stages>{}),
      cute::conditional_t<cutlass::gemm::detail::is_mn_major<StrideA>(), Step<_2, _1, _3>,
                          Step<_1, _2, _3>>{}));
  using SmemLayoutB = decltype(UMMA::tile_to_mma_shape(
      SmemLayoutAtomB{}, append(MmaShapeB_NK{}, Int<NumComputeMtxs * Stages>{}),
      cute::conditional_t<cutlass::gemm::detail::is_mn_major<StrideB>(), Step<_2, _1, _3>,
                          Step<_1, _2, _3>>{}));

  struct SharedStorage {
    struct TensorStorage : cute::aligned_struct<128, _0> {
      alignas(1024) cute::ArrayEngine<ElementA, cute::cosize_v<SmemLayoutA>> smem_A;
      alignas(1024) cute::ArrayEngine<ElementB, cute::cosize_v<SmemLayoutB>> smem_B;
    } tensors;
    struct PipelineStorage {
      alignas(16) typename MainloopABPipeline::SharedStorage pipeline_ab;
      alignas(16) typename MainloopSFPipeline::SharedStorage pipeline_sf;
      alignas(16) typename AccumulatorPipeline::SharedStorage pipeline_accum;
    };
  };
  using TensorStorage = typename SharedStorage::TensorStorage;
  using PipelineStorage = typename SharedStorage::PipelineStorage;

  // one thread of the leader CTA arms the barrier for both CTAs' three planes of A and B
  static constexpr uint32_t TmaTransactionBytes =
      NumComputeMtxs *
      (cutlass::bits_to_bytes(size(AtomThrShapeMNK{}) * cosize(take<0, 3>(SmemLayoutA{})) *
                              cute::sizeof_bits_v<ElementA>) +
       cutlass::bits_to_bytes(size(AtomThrShapeMNK{}) * cosize(take<0, 3>(SmemLayoutB{})) *
                              cute::sizeof_bits_v<ElementB>));

  template <class AccTensor>
  struct TmemStorage {
    AccTensor accumulators;
  };

  struct Arguments {
    ElementA const* ptr_A{nullptr};
    StrideA dA{};
    ElementB const* ptr_B{nullptr};
    StrideB dB{};
  };

  // the plane mode is folded into the batch mode: (M|N, K, (3, L))
  struct Params {
    using ClusterLayout_VMNK =
        decltype(tiled_divide(make_layout(ClusterShape{}), make_tile(typename TiledMma::AtomThrID{})));
    using TMA_A = decltype(make_tma_atom_A_sm100<ElementA>(
        GmemTiledCopyA{},
        make_tensor(static_cast<ElementA const*>(nullptr),
                    make_layout(make_shape(int32_t(0), int32_t(0), make_shape(int32_t(0), int32_t(0))),
                                StrideA{})),
        SmemLayoutA{}(_, _, _, cute::Int<0>{}), TileShape{}, TiledMma{}, ClusterLayout_VMNK{}));
    using TMA_B = decltype(make_tma_atom_B_sm100<ElementB>(
        GmemTiledCopyB{},
        make_tensor(static_cast<ElementB const*>(nullptr),
                    make_layout(make_shape(int32_t(0), int32_t(0), make_shape(int32_t(0), int32_t(0))),
                                StrideB{})),
        SmemLayoutB{}(_, _, _, cute::Int<0>{}), TileShape{}, TiledMma{}, ClusterLayout_VMNK{}));
    TMA_A tma_load_a;
    TMA_B tma_load_b;
  };

  CUTLASS_DEVICE
  CollectiveMma(Params const& params, ClusterShape cluster_shape, uint32_t block_rank_in_cluster)
      : cluster_shape_(cluster_shape), block_rank_in_cluster_(block_rank_in_cluster) {
    observed_tma_load_a_ = &params.tma_load_a;
    observed_tma_load_b_ = &params.tma_load_b;
  }

  template <class ProblemShape>
  static constexpr Params to_underlying_arguments(ProblemShape const& problem_shape,
                                                  Arguments const& args, void*,
                                                  cutlass::KernelHardwareInfo const& = {}) {
    auto [M, N, K, L] = append<4>(problem_shape, 1);
    Tensor tensor_a = make_tensor(
        args.ptr_A, make_layout(make_shape(M, K, make_shape(int32_t(NumComputeMtxs), L)), args.dA));
    Tensor tensor_b = make_tensor(
        args.ptr_B, make_layout(make_shape(N, K, make_shape(int32_t(NumComputeMtxs), L)), args.dB));
    auto cluster_layout_vmnk =
        tiled_divide(make_layout(ClusterShape{}), make_tile(typename TiledMma::AtomThrID{}));
    return {make_tma_atom_A_sm100<ElementA>(GmemTiledCopyA{}, tensor_a,
                                            SmemLayoutA{}(_, _, _, cute::Int<0>{}), TileShape{},
                                            TiledMma{}, cluster_layout_vmnk),
            make_tma_atom_B_sm100<ElementB>(GmemTiledCopyB{}, tensor_b,
                                            SmemLayoutB{}(_, _, _, cute::Int<0>{}), TileShape{},
                                            TiledMma{}, cluster_layout_vmnk)};
  }

  // TMA: 16-byte aligned base and strides (checked by the caller, which knows the strides)
  template <class ProblemShape>
  static bool can_implement(ProblemShape const&, Arguments const& args) {
    return (reinterpret_cast<uintptr_t>(args.ptr_A) % 16 == 0) &&
           (reinterpret_cast<uintptr_t>(args.ptr_B) % 16 == 0);
  }

  CUTLASS_DEVICE void prefetch_tma_descriptors() {
    cute::prefetch_tma_descriptor(observed_tma_load_a_->get_tma_descriptor());
    cute::prefetch_tma_descriptor(observed_tma_load_b_->get_tma_descriptor());
  }

  CUTLASS_DEVICE static auto partition_accumulator_shape() {
    return partition_shape_C(TiledMma{}, take<0, 2>(TileShape{}));
  }

  template <class EpilogueTile, bool IsOverlappingAccum = false>
  CUTLASS_DEVICE static auto init_tmem_tensors(EpilogueTile) {
    TiledMma tiled_mma;
    Tensor accumulators =
        cutlass::detail::make_sm100_accumulator<AccumulatorPipelineStageCount, IsOverlappingAccum>(
            tiled_mma, partition_accumulator_shape(), EpilogueTile{});
    TmemStorage<decltype(accumulators)> tmem_storage;
    tmem_storage.accumulators = accumulators;
    return tmem_storage;
  }

  template <class AccTensor>
  CUTLASS_DEVICE static void set_tmem_offsets(TmemStorage<AccTensor>& tmem_storage,
                                              uint32_t tmem_base_addr) {
    tmem_storage.accumulators.data() = tmem_base_addr;
  }

  template <class KTileCount, class GTensorA, class GTensorB, class STensorA, class STensorB>
  struct LoadABParams {
    KTileCount k_tiles;
    GTensorA tAgA_mkl;
    GTensorB tBgB_nkl;
    STensorA tAsA;
    STensorB tBsB;
  };

  template <class ProblemShape_MNKL, class MainloopParams>
  CUTLASS_DEVICE auto load_ab_init(ProblemShape_MNKL const& problem_shape_MNKL,
                                   MainloopParams const&, TensorStorage& shared_tensors) const {
    using X = Underscore;
    auto [M, N, K, L] = problem_shape_MNKL;
    Tensor mA_mkl = observed_tma_load_a_->get_tma_tensor(
        make_shape(M, K, make_shape(int32_t(NumComputeMtxs), L)));
    Tensor mB_nkl = observed_tma_load_b_->get_tma_tensor(
        make_shape(N, K, make_shape(int32_t(NumComputeMtxs), L)));
    Tensor gA_mkl = local_tile(mA_mkl, TileShape{}, make_coord(_, _, _), Step<_1, X, _1>{});
    Tensor gB_nkl = local_tile(mB_nkl, TileShape{}, make_coord(_, _, _), Step<X, _1, _1>{});

    ThrMMA cta_mma = TiledMma{}.get_slice(blockIdx.x % size(typename TiledMma::AtomThrID{}));
    Tensor tCgA_mkl = cta_mma.partition_A(gA_mkl);  // (MMA, MMA_M, MMA_K, m, k, (3, l))
    Tensor tCgB_nkl = cta_mma.partition_B(gB_nkl);  // (MMA, MMA_N, MMA_K, n, k, (3, l))
    Tensor sA = make_tensor(make_smem_ptr(shared_tensors.smem_A.begin()), SmemLayoutA{});
    Tensor sB = make_tensor(make_smem_ptr(shared_tensors.smem_B.begin()), SmemLayoutB{});

    Layout cta_layout_vmnk =
        tiled_divide(make_layout(cluster_shape_), make_tile(typename TiledMma::AtomThrID{}));
    auto cta_coord_vmnk = cta_layout_vmnk.get_flat_coord(block_rank_in_cluster_);
    auto [tAgA_mkl, tAsA] = tma_partition(*observed_tma_load_a_, get<2>(cta_coord_vmnk),
                                          make_layout(size<2>(cta_layout_vmnk)),
                                          group_modes<0, 3>(sA), group_modes<0, 3>(tCgA_mkl));
    auto [tBgB_nkl, tBsB] = tma_partition(*observed_tma_load_b_, get<1>(cta_coord_vmnk),
                                          make_layout(size<1>(cta_layout_vmnk)),
                                          group_modes<0, 3>(sB), group_modes<0, 3>(tCgB_nkl));
    return LoadABParams<decltype(shape<3>(gA_mkl)), decltype(tAgA_mkl), decltype(tBgB_nkl),
                        decltype(tAsA), decltype(tBsB)>{shape<3>(gA_mkl), tAgA_mkl, tBgB_nkl,
                                                        tAsA, tBsB};
  }

  struct LoadSFParams {
    int k_tiles;
  };
  template <class ProblemShape_MNKL, class MainloopParams>
  CUTLASS_DEVICE auto load_sf_init(ProblemShape_MNKL const& problem_shape_MNKL,
                                   MainloopParams const&, TensorStorage&) const {
    return LoadSFParams{int(ceil_div(get<2>(problem_shape_MNKL), size<2>(TileShape{})))};
  }

  template <class MmaA, class MmaB>
  struct MmaParams {
    MmaA tCrA;
    MmaB tCrB;
  };
  template <class AccTensor>
  CUTLASS_DEVICE auto mma_init(TmemStorage<AccTensor>, TensorStorage& shared_tensors) const {
    Tensor sA = make_tensor(make_smem_ptr(shared_tensors.smem_A.begin()), SmemLayoutA{});
    Tensor sB = make_tensor(make_smem_ptr(shared_tensors.smem_B.begin()), SmemLayoutB{});
    Tensor tCrA = TiledMma::make_fragment_A(sA);  // (MMA, MMA_M, MMA_K, PLANE + 3 * PIPE)
    Tensor tCrB = TiledMma::make_fragment_B(sB);  // (MMA, MMA_N, MMA_K, PLANE + 3 * PIPE)
    return MmaParams<decltype(tCrA), decltype(tCrB)>{tCrA, tCrB};
  }

  template <class ProblemShape_MNKL>
  CUTLASS_DEVICE auto accum_init(ProblemShape_MNKL const&, TensorStorage&) const {
    return 0;
  }

  // TMA producer: the three planes of A and of B for each k-block
  template <class LoadABParams, class TileCoordMNKL, class KTileIterator>
  CUTLASS_DEVICE auto load_ab(MainloopABPipeline pipeline, MainloopABPipelineState state,
                              LoadABParams const& load_inputs, TileCoordMNKL const& cta_coord_mnkl,
                              KTileIterator k_tile_iter, int k_tile_count) {
    Tensor tAgA = load_inputs.tAgA_mkl(
        _, get<0>(cta_coord_mnkl) / size(typename TiledMma::AtomThrID{}), _, _);  // (TMA, k, (3, l))
    Tensor tBgB = load_inputs.tBgB_nkl(_, get<1>(cta_coord_mnkl), _, _);
    int const l = get<3>(cta_coord_mnkl);
    auto barrier_token = pipeline.producer_try_acquire(state);
    CUTLASS_PRAGMA_NO_UNROLL
    while (k_tile_count > 0) {
      pipeline.producer_acquire(state, barrier_token);
      using BarrierType = typename MainloopABPipeline::ProducerBarrierType;
      BarrierType* tma_barrier = pipeline.producer_get_barrier(state);
      int const write_stage = state.index();
      ++state;
      barrier_token = pipeline.producer_try_acquire(state);
      if (cute::elect_one_sync()) {
        CUTLASS_PRAGMA_UNROLL
        for (int p = 0; p < NumComputeMtxs; ++p) {
          copy(observed_tma_load_a_->with(*tma_barrier), tAgA(_, *k_tile_iter, make_coord(p, l)),
               load_inputs.tAsA(_, write_stage * NumComputeMtxs + p));
          copy(observed_tma_load_b_->with(*tma_barrier), tBgB(_, *k_tile_iter, make_coord(p, l)),
               load_inputs.tBsB(_, write_stage * NumComputeMtxs + p));
        }
      }
      --k_tile_count;
      ++k_tile_iter;
    }
    return cute::make_tuple(state, k_tile_iter);
  }

  CUTLASS_DEVICE void load_ab_tail(MainloopABPipeline pipeline, MainloopABPipelineState state) {
    pipeline.producer_tail(state);
  }

  template <class LoadSFParams, class TileCoordMNKL, class KTileIterator>
  CUTLASS_DEVICE auto load_sf(MainloopSFPipeline, MainloopSFPipelineState state, LoadSFParams const&,
                              TileCoordMNKL const&, KTileIterator k_tile_iter, int) {
    return cute::make_tuple(state, k_tile_iter);
  }
  CUTLASS_DEVICE void load_sf_tail(MainloopSFPipeline, MainloopSFPipelineState) {}

  // MMA warp: the emulated collective's band order, scaling and promotion interval, unchanged
  template <class TmemStorage, class MmaParams, class CtaTileCoord>
  CUTLASS_DEVICE auto mma(cute::tuple<MainloopABPipeline, AccumulatorPipeline> pipelines,
                          cute::tuple<MainloopABPipelineState, AccumulatorPipelineState> states,
                          TmemStorage tmem_storage, MmaParams const& mma_inputs, CtaTileCoord,
                          int k_tile_count) {
    TiledMma tiled_mma;
    auto [mainloop_pipeline, accumulator_pipeline] = pipelines;
    auto [mainloop_state, acc_state] = states;
    auto const& tCrA = mma_inputs.tCrA;
    auto const& tCrB = mma_inputs.tCrB;
    using ZeroScaler = cute::integral_constant<uint32_t, 0>;
    using Scaler = cute::integral_constant<uint32_t, ScalingFactor>;
    constexpr int PI = AccPromotionInterval;

    uint32_t skip_wait = k_tile_count <= 0;
    auto barrier_token = mainloop_pipeline.consumer_try_wait(mainloop_state, skip_wait);
    CUTLASS_PRAGMA_NO_UNROLL
    while (k_tile_count > 0) {
      mainloop_pipeline.consumer_wait(mainloop_state, barrier_token);
      int const s = mainloop_state.index() * NumComputeMtxs;
      auto curr_mainloop_state = mainloop_state;
      ++mainloop_state;
      --k_tile_count;
      skip_wait = k_tile_count <= 0;
      barrier_token = mainloop_pipeline.consumer_try_wait(mainloop_state, skip_wait);

      auto tCrA0 = tCrA(_, _, _, s + 0);
      auto tCrA1 = tCrA(_, _, _, s + 1);
      auto tCrA2 = tCrA(_, _, _, s + 2);
      auto tCrB0 = tCrB(_, _, _, s + 0);
      auto tCrB1 = tCrB(_, _, _, s + 1);
      auto tCrB2 = tCrB(_, _, _, s + 2);

      CUTLASS_PRAGMA_UNROLL
      for (int k_block = 0; k_block < size<2>(tCrA); k_block += PI) {
        accumulator_pipeline.producer_acquire(acc_state);
        auto tCtC = tmem_storage.accumulators(_, _, _, acc_state.index());
        auto accumulate = UMMA::ScaleOut::Zero;
        if constexpr (NumBandsToCompute == 5) {
          cute::gemm(tiled_mma.with(accumulate, ZeroScaler{}), tCrA2(_, _, k_block), tCrB2(_, _, k_block), tCtC);
          accumulate = UMMA::ScaleOut::One;
          CUTLASS_PRAGMA_UNROLL
          for (int t = 1; t < PI; t++) {
            cute::gemm(tiled_mma.with(accumulate, ZeroScaler{}), tCrA2(_, _, k_block + t), tCrB2(_, _, k_block + t), tCtC);
          }
        }
        if constexpr (NumBandsToCompute >= 4) {
          cute::gemm(tiled_mma.with(accumulate, Scaler{}), tCrA1(_, _, k_block), tCrB2(_, _, k_block), tCtC);
          accumulate = UMMA::ScaleOut::One;
          cute::gemm(tiled_mma.with(accumulate, ZeroScaler{}), tCrA2(_, _, k_block), tCrB1(_, _, k_block), tCtC);
          CUTLASS_PRAGMA_UNROLL
          for (int t = 1; t < PI; t++) {
            cute::gemm(tiled_mma.with(accumulate, ZeroScaler{}), tCrA1(_, _, k_block + t), tCrB2(_, _, k_block + t), tCtC);
            cute::gemm(tiled_mma.with(accumulate, ZeroScaler{}), tCrA2(_, _, k_block + t), tCrB1(_, _, k_block + t), tCtC);
          }
        }
        // band 3: x0*y2, x1*y1, x2*y0
        cute::gemm(tiled_mma.with(accumulate, Scaler{}), tCrA0(_, _, k_block), tCrB2(_, _, k_block), tCtC);
        accumulate = UMMA::ScaleOut::One;
        cute::gemm(tiled_mma.with(accumulate, ZeroScaler{}), tCrA1(_, _, k_block), tCrB1(_, _, k_block), tCtC);
        cute::gemm(tiled_mma.with(accumulate, ZeroScaler{}), tCrA2(_, _, k_block), tCrB0(_, _, k_block), tCtC);
        CUTLASS_PRAGMA_UNROLL
        for (int t = 1; t < PI; t++) {
          cute::gemm(tiled_mma.with(accumulate, ZeroScaler{}), tCrA0(_, _, k_block + t), tCrB2(_, _, k_block + t), tCtC);
          cute::gemm(tiled_mma.with(accumulate, ZeroScaler{}), tCrA1(_, _, k_block + t), tCrB1(_, _, k_block + t), tCtC);
          cute::gemm(tiled_mma.with(accumulate, ZeroScaler{}), tCrA2(_, _, k_block + t), tCrB0(_, _, k_block + t), tCtC);
        }
        // band 2: x0*y1, x1*y0
        cute::gemm(tiled_mma.with(accumulate, Scaler{}), tCrA0(_, _, k_block), tCrB1(_, _, k_block), tCtC);
        cute::gemm(tiled_mma.with(accumulate, ZeroScaler{}), tCrA1(_, _, k_block), tCrB0(_, _, k_block), tCtC);
        CUTLASS_PRAGMA_UNROLL
        for (int t = 1; t < PI; t++) {
          cute::gemm(tiled_mma.with(accumulate, ZeroScaler{}), tCrA0(_, _, k_block + t), tCrB1(_, _, k_block + t), tCtC);
          cute::gemm(tiled_mma.with(accumulate, ZeroScaler{}), tCrA1(_, _, k_block + t), tCrB0(_, _, k_block + t), tCtC);
        }
        // band 1: x0*y0
        cute::gemm(tiled_mma.with(accumulate, Scaler{}), tCrA0(_, _, k_block), tCrB0(_, _, k_block), tCtC);
        CUTLASS_PRAGMA_UNROLL
        for (int t = 1; t < PI; t++) {
          cute::gemm(tiled_mma.with(accumulate, ZeroScaler{}), tCrA0(_, _, k_block + t), tCrB0(_, _, k_block + t), tCtC);
        }
        accumulator_pipeline.producer_commit(acc_state);
        ++acc_state;
      }
      mainloop_pipeline.consumer_release(curr_mainloop_state);
    }
    return cute::make_tuple(mainloop_state, acc_state);
  }

  // epilogue warps: promote each TMEM accumulator stage into fp32 registers (acc += stage)
  template <class AccumParams, class TmemStorage, class CtaTileCoord, class CopyOpT2R, class EpilogueTile>
  CUTLASS_DEVICE auto accum(cute::tuple<AccumulatorPipeline, MainloopSFPipeline> pipelines,
                            cute::tuple<AccumulatorPipelineState, MainloopSFPipelineState> states,
                            TmemStorage tmem_storage, AccumParams const&, CtaTileCoord, CopyOpT2R,
                            EpilogueTile, int k_tile_count) {
    auto [accumulator_pipeline, sf_pipeline] = pipelines;
    auto [acc_state, sf_state] = states;

    Tensor tAcc = tmem_storage.accumulators(make_coord(_, _), _0{}, _0{}, _0{});
    Tensor tAcc_epi = flat_divide(tAcc, EpilogueTile{});  // (EPI_TILE_M, EPI_TILE_N, EPI_M, EPI_N)
    TiledCopy tiled_t2r = make_tmem_copy(CopyOpT2R{}, tAcc_epi(_, _, _0{}, _0{}));
    ThrCopy thread_t2r = tiled_t2r.get_slice(threadIdx.x % size(tiled_t2r));
    Tensor tTR_rGlobAcc = make_tensor<ElementAccumulator>(shape(thread_t2r.partition_D(tAcc_epi)));
    Tensor tTR_rAcc = make_tensor<ElementAccumulator>(shape(tTR_rGlobAcc(_, _, _, _0{}, _0{})));
    clear(tTR_rGlobAcc);

    CUTLASS_PRAGMA_NO_UNROLL
    for (int n = k_tile_count * StagesPerTile; n > 0; --n) {
      accumulator_pipeline.consumer_wait(acc_state);
      Tensor tStage = tmem_storage.accumulators(make_coord(_, _), _0{}, _0{}, acc_state.index());
      Tensor tTR_tAcc = thread_t2r.partition_S(flat_divide(tStage, EpilogueTile{}));
      CUTLASS_PRAGMA_UNROLL
      for (int epi_m = 0; epi_m < size<2>(tAcc_epi); ++epi_m) {
        CUTLASS_PRAGMA_UNROLL
        for (int epi_n = 0; epi_n < size<3>(tAcc_epi); ++epi_n) {
          copy(tiled_t2r, tTR_tAcc(_, _, _, epi_m, epi_n), tTR_rAcc);
          Tensor g = tTR_rGlobAcc(_, _, _, epi_m, epi_n);
          CUTLASS_PRAGMA_UNROLL
          for (int i = 0; i < size(tTR_rAcc); ++i) g(i) = g(i) + tTR_rAcc(i);
        }
      }
      cutlass::arch::fence_view_async_tmem_load();
      accumulator_pipeline.consumer_release(acc_state);
      ++acc_state;
    }
    return cute::make_tuple(tTR_rGlobAcc, tiled_t2r, cute::make_tuple(acc_state, sf_state));
  }

 protected:
  typename Params::TMA_A const* observed_tma_load_a_ = nullptr;
  typename Params::TMA_B const* observed_tma_load_b_ = nullptr;
  ClusterShape cluster_shape_;
  uint32_t block_rank_in_cluster_;
};

}  // namespace cutlass::gemm::collective
