// K4 — DLRM pairwise dot interaction, optionally fused with the embedding gather.
//
// The reference's DLRM.call concatenates instead of interacting (src/ctr/dlrm/model.py:48) and
// cites arXiv 1906.00091 (:7); SURVEY.md §8 a5 defines the op from the paper:
//   X = stack([bottom_mlp(dense), e_1 .. e_F])  (B, F1, D),  Z = X X^T,
//   out = concat([X[:,0,:], Z[i,j] for i > j (row-major lower triangle)])   (B, D + F1(F1-1)/2)
//
// One warp owns one sample at a time.  Its F1 rows are staged in shared memory by the TMA
// engine — one cp.async.bulk (SASS UBLKCP) per row, straight from the embedding tables when
// fused, so gathered rows never round-trip HBM — completing on a per-warp mbarrier.  The
// Gram matrix is computed in fp32 FFMA with 4x4 register blocks (lane <-> block of the lower
// triangle); rows of a block are interleaved with stride F1p/4 so the 128-bit shared loads of
// a warp hit distinct banks.  Backward re-gathers X (cheaper than saving it) and forms
// dX = (S + S^T) X with lanes owning 4 embedding columns each.
// Bound: HBM (ids + rows in, D+P floats out) with the fp32 FMA pipe close behind (DESIGN.md).
#include <type_traits>

#include "rtf_common.cuh"

namespace rtf {

struct DotParams {
  const float* table[RTF_MAX_FIELDS];  // gather mode: row i >= 1 comes from table[i-1]
  long long rows[RTF_MAX_FIELDS];
  const void* ids;
  long long ids_sb, ids_sf;
  int gather;  // 1: rows 1.. come from table[i-1][ids]; 0: every row i is rbase[i] + b*rstride[i]
  const float* rbase[RTF_MAX_FIELDS];  // row sources (row 0 always; all rows when !gather)
  long long rstride[RTF_MAX_FIELDS];
  float* gbase[RTF_MAX_FIELDS];  // bwd: where dX row i of sample b goes: gbase[i] + b*gstride[i]
  long long gstride[RTF_MAX_FIELDS];
  long long B;
  int F1, D, out_cols;
  float* out;  // fwd (B, out_cols...)
  long long out_sb;
  const float* gout;  // bwd
  long long gout_sb;
  float* xsave;  // fwd, optional: rows 1..F1-1 of every sample copied to (B, (F1-1)*D) — lets a
  long long xsave_sb;  // backward re-read rows locally when the forward pulled them over NVLink
  // tables sharded over G GPUs, addressed through NVLink peer pointers (device arrays [F][G]):
  // field f is row-wise sharded if bit f of rw_mask is set (row r lives on rank r % G at local
  // row r / G), else wholly on one rank whose pointer sits in entry [f][0].
  const long long* peer_tab;   // fwd: table shard base pointers (or owner-gathered row buffers)
  const long long* peer_str;   // fwd, optional: rows were gathered by their owners into per-rank
                               // (B_global, T_g*D) buffers; entry = elements between samples and
                               // peer_tab entry = base of the field's column in that buffer
  const long long* peer_gptr;  // bwd: where dX rows go: base of field f's column in rank g's buffer
  const long long* peer_gstr;  // bwd: elements between consecutive samples in that buffer
  unsigned long long rw_mask;
  long long sample0;           // bwd: global index of this rank's first sample
  int peer_G;
  int32_t* err;
};

__device__ __forceinline__ void peer_split(const DotParams& P, int f, long long id, int& g,
                                           long long& row) {
  if ((P.rw_mask >> f) & 1ull) {
    g = (int)(id % P.peer_G);
    row = id / P.peer_G;
  } else {
    g = 0;
    row = id;
  }
}

__host__ __device__ inline int dot_row_stride(int D) { return D + ((D % 8 == 0) ? 4 : 8); }

template <typename IdT>
__device__ __forceinline__ const float* dot_src_row(const DotParams& P, long long b, int i) {
  if (!P.gather || i == 0) return P.rbase[i] + b * P.rstride[i];
  const long long id = load_id((const IdT*)P.ids, b * P.ids_sb + (long long)(i - 1) * P.ids_sf,
                               P.rows[i - 1], P.err);
  if (id < 0) return nullptr;
  if (P.peer_tab) {
    int g;
    long long row;
    peer_split(P, i - 1, id, g, row);
    const int e = (i - 1) * P.peer_G + g;
    if (P.peer_str)  // pull by sample from the holder's gathered rows (sequential addresses)
      return reinterpret_cast<const float*>(P.peer_tab[e]) + (P.sample0 + b) * P.peer_str[e];
    return reinterpret_cast<const float*>(P.peer_tab[e]) + row * P.D;  // pull from the table shard
  }
  return P.table[i - 1] + id * P.D;
}

// stage the F1 rows of sample b into xt (row stride RS) with bulk async copies
template <typename IdT>
__device__ __forceinline__ void dot_issue_rows(const DotParams& P, long long b, float* xt, int RS,
                                               uint64_t* bar, int lane) {
  const int F1 = P.F1, D = P.D;
  const float* src[2];
  unsigned nvalid = 0;
#pragma unroll
  for (int k = 0; k < 2; ++k) {
    const int r = lane + 32 * k;
    src[k] = r < F1 ? dot_src_row<IdT>(P, b, r) : nullptr;
    if (r < F1 && !src[k])
      for (int d = 0; d < D; ++d) xt[r * RS + d] = 0.f;  // bad id: row reads as zeros
    nvalid += __popc(__ballot_sync(0xffffffffu, src[k] != nullptr));
  }
  if (lane == 0) mbar_expect_tx(bar, nvalid * (unsigned)D * 4u);
  __syncwarp();
#pragma unroll
  for (int k = 0; k < 2; ++k) {
    const int r = lane + 32 * k;
    if (src[k]) bulk_g2s(xt + r * RS, src[k], (unsigned)D * 4u, bar);
  }
}

// The same in two steps: ids -> row sources of sample b (lane owns rows lane and lane + 32) without
// touching shared memory, then the copies.  A warp resolves the NEXT sample's addresses (a dependent
// global load, ~1 us) before its FMA loop and issues the copies the moment the tile is free, instead
// of paying the id load in front of every gather.
template <typename IdT>
__device__ __forceinline__ void dot_resolve_rows(const DotParams& P, long long b, int lane,
                                                 const float* (&src)[2]) {
#pragma unroll
  for (int k = 0; k < 2; ++k) {
    const int r = lane + 32 * k;
    src[k] = r < P.F1 ? dot_src_row<IdT>(P, b, r) : nullptr;
  }
}
__device__ __forceinline__ void dot_issue_resolved(const DotParams& P, float* xt, int RS,
                                                   uint64_t* bar, int lane,
                                                   const float* const (&src)[2]) {
  const int F1 = P.F1, D = P.D;
  unsigned nvalid = 0;
#pragma unroll
  for (int k = 0; k < 2; ++k) {
    const int r = lane + 32 * k;
    if (r < F1 && !src[k])
      for (int d = 0; d < D; ++d) xt[r * RS + d] = 0.f;  // bad id: row reads as zeros
    nvalid += __popc(__ballot_sync(0xffffffffu, src[k] != nullptr));
  }
  if (lane == 0) mbar_expect_tx(bar, nvalid * (unsigned)D * 4u);
  __syncwarp();
#pragma unroll
  for (int k = 0; k < 2; ++k) {
    const int r = lane + 32 * k;
    if (src[k]) bulk_g2s(xt + r * RS, src[k], (unsigned)D * 4u, bar);
  }
}

__device__ __forceinline__ void tri_block(int blk, int& bi, int& bj) {
  // blk -> (bi, bj), bj <= bi, row-major over the lower triangle of blocks
  int i = (int)((sqrtf(8.f * blk + 1.f) - 1.f) * 0.5f);
  while ((i + 1) * (i + 2) / 2 <= blk) ++i;
  while (i * (i + 1) / 2 > blk) --i;
  bi = i;
  bj = blk - i * (i + 1) / 2;
}

template <typename IdT>
__global__ void __launch_bounds__(512, 1)
dot_fwd_kernel(const __grid_constant__ DotParams P, int warp_floats) {
  extern __shared__ __align__(16) float smem[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
  const int F1 = P.F1, D = P.D;
  const int F1p = (F1 + 3) & ~3, nbr = F1p >> 2;
  const int RS = dot_row_stride(D);
  const int npairs = F1 * (F1 - 1) / 2;
  float* xt = smem + (size_t)warp * warp_floats;
  float* zst = xt + F1p * RS;
  uint64_t* bar = reinterpret_cast<uint64_t*>(zst + ((npairs + 3) & ~3));

  if (lane == 0) {
    mbar_init(bar, 1);
    mbar_fence_init();
  }
  for (int i = F1 * RS + lane; i < F1p * RS; i += 32) xt[i] = 0.f;  // pad rows stay zero
  __syncwarp();

  const long long stride = (long long)gridDim.x * nwarps;
  long long b = (long long)blockIdx.x * nwarps + warp;
  uint32_t parity = 0;
  if (b < P.B) dot_issue_rows<IdT>(P, b, xt, RS, bar, lane);
  const int nblk = nbr * (nbr + 1) / 2;

  for (; b < P.B; b += stride) {
    mbar_wait(bar, parity);
    parity ^= 1;
    for (int blk = lane; blk < nblk; blk += 32) {
      int bi, bj;
      tri_block(blk, bi, bj);
      // block (bi,bj) covers rows {bi + r*nbr} x {bj + c*nbr}
      // packed fp32x2 FMAs (sm_100 FFMA2): half the issue slots of scalar FFMA; the two halves
      // of a pair accumulate even / odd pairs of d and are added at the end
      float2 acc[4][4];
#pragma unroll
      for (int r = 0; r < 4; ++r)
#pragma unroll
        for (int c = 0; c < 4; ++c) acc[r][c] = make_float2(0.f, 0.f);
      const float* pa = xt + bi * RS;
      const float* pb = xt + bj * RS;
      const int rstep = nbr * RS;
#pragma unroll 2
      for (int d = 0; d < D; d += 4) {
        float4 a[4], q[4];
#pragma unroll
        for (int r = 0; r < 4; ++r) {
          a[r] = *reinterpret_cast<const float4*>(pa + r * rstep + d);
          q[r] = *reinterpret_cast<const float4*>(pb + r * rstep + d);
        }
#pragma unroll
        for (int r = 0; r < 4; ++r)
#pragma unroll
          for (int c = 0; c < 4; ++c) {
            acc[r][c] = __ffma2_rn(make_float2(a[r].x, a[r].y), make_float2(q[c].x, q[c].y), acc[r][c]);
            acc[r][c] = __ffma2_rn(make_float2(a[r].z, a[r].w), make_float2(q[c].z, q[c].w), acc[r][c]);
          }
      }
#pragma unroll
      for (int r = 0; r < 4; ++r)
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          const int i = bi + r * nbr, j = bj + c * nbr;
          const float z = acc[r][c].x + acc[r][c].y;
          if (i < F1 && j < i) zst[i * (i - 1) / 2 + j] = z;
          else if (bi != bj && j < F1 && i < j) zst[j * (j - 1) / 2 + i] = z;
        }
    }
    __syncwarp();
    float* o = P.out + b * P.out_sb;
    for (int d = lane; d < D; d += 32) o[d] = xt[d];
    for (int p = lane; p < npairs; p += 32) o[D + p] = zst[p];
    for (int p = D + npairs + lane; p < P.out_cols; p += 32) o[p] = 0.f;
    if (P.xsave) {
      float* xs = P.xsave + b * P.xsave_sb;
      const int nv = D >> 2;
      for (int e = lane; e < (F1 - 1) * nv; e += 32) {
        const int r = e / nv, c = e - r * nv;
        *reinterpret_cast<float4*>(xs + r * D + 4 * c) =
            *reinterpret_cast<const float4*>(xt + (r + 1) * RS + 4 * c);
      }
    }
    __syncwarp();  // every lane is done reading xt/zst before the next sample overwrites them
    if (b + stride < P.B) dot_issue_rows<IdT>(P, b + stride, xt, RS, bar, lane);
  }
}

// Forward, 7x7 register blocks.  The 4x4 kernel above is bound by shared-memory wavefronts (ncu,
// profiles/r2_ncu_full_summary.txt: 71 M wavefronts; with the row gather switched off it still
// takes 0.30 of its 0.37 ms, with the Gram loop switched off 0.12): a lane loads 8 float4 per 32
// packed FMAs, and a shared load costs wavefronts by the bytes each lane receives, broadcast or
// not.  Here a lane owns a 7x7 block of the Gram matrix (rows {bi + r*nbr} x {bj + c*nbr}: 10
// blocks of the lower triangle for 22..28 rows) and the lanes left over split the embedding
// dimension: lane = (block, d-group), d-group g takes the float2 columns g, g + G, ... (G = 32 /
// blocks = 3).  14 float2 loads feed 49 packed FMAs: 0.57 wavefronts per FMA2 instead of 1.0.
// The G partial blocks are added in group order with two shuffles (deterministic) and group 0
// stores its block into a square Z tile with immediate offsets — no per-element branches; the
// packed lower triangle is read back through a (p -> position) table.  The next sample's row
// gather is issued as soon as the Gram loop has read the rows, under the reduction and stores.
// D and the block-row count are template parameters so that the 14 shared-memory addresses of an
// iteration are immediates off two base registers (runtime strides cost 14 address registers and
// made ptxas reload q[c] into one register: 0.70 ms).  Bank map: word = row*(D+4) + 2e, the 16
// lanes of a half-warp read (2 row + e) mod 16 distinct or identical addresses — conflict-free.
template <typename IdT, int D, int nbr>
__global__ void __launch_bounds__(384, 1)
dot_fwd7_kernel(const __grid_constant__ DotParams P, int warp_floats) {
  extern __shared__ __align__(16) float smem[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
  const int F1 = P.F1;
  constexpr int F1p = nbr * 7;
  constexpr int RS = D + ((D % 8 == 0) ? 4 : 8);
  constexpr int ZS = F1p + 1;
  const int npairs = F1 * (F1 - 1) / 2;
  constexpr int nblk = nbr * (nbr + 1) / 2;
  constexpr int ngrp = 32 / nblk;
  const int blk = lane % nblk, grp = lane / nblk;    // grp >= ngrp: spare lane
  // CTA-shared pair table, then per-warp regions
  unsigned short* pair_ij = reinterpret_cast<unsigned short*>(smem);
  const int pair_floats = ((npairs + 1) / 2 + 3) & ~3;
  float* xt = smem + pair_floats + (size_t)warp * warp_floats;   // [F1p][RS]
  float* Z = xt + F1p * RS;                                      // [F1p][ZS]
  uint64_t* bar = reinterpret_cast<uint64_t*>(Z + ((F1p * ZS + 3) & ~3));
  int bi, bj;
  tri_block(blk, bi, bj);

  for (int p = threadIdx.x; p < npairs; p += blockDim.x) {
    int i = (int)((1.f + sqrtf(1.f + 8.f * p)) * 0.5f);
    while (i * (i - 1) / 2 > p) --i;
    while ((i + 1) * i / 2 <= p) ++i;
    // pair (i, j), i > j, is computed by block (max, min) of (i % nbr, j % nbr) and lands at
    // Z[i][j] when i's block row is the larger one, else at Z[j][i]
    const int j = p - i * (i - 1) / 2;
    pair_ij[p] = (unsigned short)((i % nbr >= j % nbr) ? i * ZS + j : j * ZS + i);
  }
  if (lane == 0) {
    mbar_init(bar, 1);
    mbar_fence_init();
  }
  for (int i = F1 * RS + lane; i < F1p * RS; i += 32) xt[i] = 0.f;  // pad rows stay zero
  __syncthreads();

  const long long stride = (long long)gridDim.x * nwarps;
  long long b = (long long)blockIdx.x * nwarps + warp;
  uint32_t parity = 0;
  if (b < P.B) dot_issue_rows<IdT>(P, b, xt, RS, bar, lane);
  constexpr int rstep = nbr * RS;
  constexpr int nd2 = D >> 1;
  const float* pa = xt + bi * RS;
  const float* pb = xt + bj * RS;
  float* zd = Z + bi * ZS + bj;      // Z[i][j]

  for (; b < P.B; b += stride) {
    mbar_wait(bar, parity);
    parity ^= 1;
    const bool more = b + stride < P.B;
    const float* src[2] = {nullptr, nullptr};
    if (more) dot_resolve_rows<IdT>(P, b + stride, lane, src);   // id loads fly under the Gram loop
    float2 acc[7][7];
#pragma unroll
    for (int r = 0; r < 7; ++r)
#pragma unroll
      for (int c = 0; c < 7; ++c) acc[r][c] = make_float2(0.f, 0.f);
    if (grp < ngrp) {
#pragma unroll 1
      for (int e = grp; e < nd2; e += ngrp) {
        float2 a[7], q[7];
#pragma unroll
        for (int r = 0; r < 7; ++r) {
          a[r] = *reinterpret_cast<const float2*>(pa + r * rstep + 2 * e);
          q[r] = *reinterpret_cast<const float2*>(pb + r * rstep + 2 * e);
        }
#pragma unroll
        for (int r = 0; r < 7; ++r)
#pragma unroll
          for (int c = 0; c < 7; ++c) acc[r][c] = __ffma2_rn(a[r], q[c], acc[r][c]);
      }
    }
    // row 0 (passed through) and the optional row copy are the last readers of xt: take them
    // now, so the next sample's gather runs under the reduction / store phase below
    float x0[(D + 31) / 32];
#pragma unroll
    for (int k = 0; k < (D + 31) / 32; ++k) x0[k] = lane + 32 * k < D ? xt[lane + 32 * k] : 0.f;
    if (P.xsave) {
      float* xs = P.xsave + b * P.xsave_sb;
      constexpr int nv = D >> 2;
      for (int e = lane; e < (F1 - 1) * nv; e += 32) {
        const int r = e / nv, c = e - r * nv;
        *reinterpret_cast<float4*>(xs + r * D + 4 * c) =
            *reinterpret_cast<const float4*>(xt + (r + 1) * RS + 4 * c);
      }
    }
    __syncwarp();  // every lane is done reading xt
    if (more) dot_issue_resolved(P, xt, RS, bar, lane, src);
    // d-group partials -> group 0, added in group order
    float z[7][7];
#pragma unroll
    for (int r = 0; r < 7; ++r)
#pragma unroll
      for (int c = 0; c < 7; ++c) {
        const float part = acc[r][c].x + acc[r][c].y;
        z[r][c] = part;
#pragma unroll
        for (int g = 1; g < ngrp; ++g) z[r][c] += __shfl_down_sync(0xffffffffu, part, g * nblk);
      }
    if (grp == 0) {     // Z[i][j], i = bi + r nbr, j = bj + c nbr (either triangle; see pair_ij)
#pragma unroll
      for (int r = 0; r < 7; ++r)
#pragma unroll
        for (int c = 0; c < 7; ++c) zd[r * (nbr * ZS) + c * nbr] = z[r][c];
    }
    __syncwarp();
    float* o = P.out + b * P.out_sb;
#pragma unroll
    for (int k = 0; k < (D + 31) / 32; ++k)
      if (lane + 32 * k < D) o[lane + 32 * k] = x0[k];
    for (int p = lane; p < npairs; p += 32) o[D + p] = Z[pair_ij[p]];
    for (int p = D + npairs + lane; p < P.out_cols; p += 32) o[p] = 0.f;
    __syncwarp();  // every lane is done reading Z before the next sample overwrites it
  }
}

// backward: dX[i] = sum_j S[i][j] X[j],  S symmetric from dZ, plus the passthrough on row 0
// row pairs of the t-th 8-row tile of an F1-row sample (the last tile only the pairs that exist)
__host__ __device__ constexpr int bwd_tile_rpn(int f1, int t) {
  return (f1 - 8 * t) > 6 ? 4 : (f1 - 8 * t) > 4 ? 3 : (f1 - 8 * t) > 2 ? 2 : 1;
}

// CF1 / CD: compile-time row count and embedding width (0 = runtime).  The kernel issues ~4 000
// instructions per sample of which 1 512 are FFMA2 (ncu: issue slots 50 %, nothing else near a
// limit), so for the shape the bench and the reference's Criteo DLRM use the loop bounds, shared-
// memory strides and tile dispatch are constants: the j loops unroll fully onto immediate offsets.
template <typename IdT, int CF1 = 0, int CD = 0>
__global__ void __launch_bounds__(CF1 ? 384 : 512, 1)   // the compile-time shape runs 12 warps (shared memory)
dot_bwd_kernel(const __grid_constant__ DotParams P, int warp_floats) {
  extern __shared__ __align__(16) float smem[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
  const int F1 = CF1 ? CF1 : P.F1, D = CD ? CD : P.D;
  const int F1p = (F1 + 7) & ~7;  // i-tiles of 8 rows
  const int SS = F1p + 4;         // S row stride: the mirrored writes S[j][i] of consecutive j would
                                  // all hit one bank with a stride of 32
  const int RS = dot_row_stride(D);
  const int npairs = F1 * (F1 - 1) / 2;
  // CTA-shared pair table, then per-warp regions
  unsigned short* pair_ij = reinterpret_cast<unsigned short*>(smem);
  const int pair_floats = ((npairs + 1) / 2 + 3) & ~3;
  float* wbase = smem + pair_floats + (size_t)warp * warp_floats;
  float* xt = wbase;                // [F1][RS]
  float* S = xt + F1 * RS;          // [F1][SS]
  uint64_t* bar = reinterpret_cast<uint64_t*>(S + F1 * SS);
  long long* ids_w = reinterpret_cast<long long*>(bar + 2);  // [64] ids of this sample (peer bwd)

  for (int p = threadIdx.x; p < npairs; p += blockDim.x) {
    int i = (int)((1.f + sqrtf(1.f + 8.f * p)) * 0.5f);
    while (i * (i - 1) / 2 > p) --i;
    while ((i + 1) * i / 2 <= p) ++i;
    pair_ij[p] = (unsigned short)((i << 8) | (p - i * (i - 1) / 2));
  }
  if (lane == 0) {
    mbar_init(bar, 1);
    mbar_fence_init();
  }
  for (int i = lane; i < F1 * SS; i += 32) S[i] = 0.f;  // diagonal and padding stay zero
  __syncthreads();

  const long long stride = (long long)gridDim.x * nwarps;
  long long b = (long long)blockIdx.x * nwarps + warp;
  uint32_t parity = 0;
  if (b < P.B) dot_issue_rows<IdT>(P, b, xt, RS, bar, lane);
  // the incoming gradient of the NEXT sample is fetched into registers while this one is being
  // processed (its HBM latency was a serial 0.07 ms in front of every sample's S fill)
  constexpr int PF = 12;                     // covers F1 <= 28; longer tails are loaded in place
  float gpre[PF];
  float4 g0pre = make_float4(0.f, 0.f, 0.f, 0.f);
  const bool g_vec = (P.gout_sb & 3) == 0 && (reinterpret_cast<uintptr_t>(P.gout) & 15) == 0;
  auto prefetch = [&](long long bb) {
    const float* gg = P.gout + bb * P.gout_sb;
#pragma unroll
    for (int q = 0; q < PF; ++q) gpre[q] = lane + 32 * q < npairs ? __ldg(gg + D + lane + 32 * q) : 0.f;
    if (lane * 4 < D) {
      if (g_vec) g0pre = __ldg(reinterpret_cast<const float4*>(gg + lane * 4));
      else g0pre = make_float4(__ldg(gg + lane * 4), __ldg(gg + lane * 4 + 1), __ldg(gg + lane * 4 + 2),
                               __ldg(gg + lane * 4 + 3));
    }
  };
  if (b < P.B) prefetch(b);

  for (; b < P.B; b += stride) {
    const float* g = P.gout + b * P.gout_sb;
    if (P.peer_gptr)  // ids decide which GPU a row-wise sharded field's gradient row goes to
      for (int f = lane; f < F1 - 1; f += 32) {
        long long id = (long long)__ldg((const IdT*)P.ids + b * P.ids_sb + (long long)f * P.ids_sf);
        ids_w[f] = (id < 0 || id >= P.rows[f]) ? -1 : id;
      }
#pragma unroll
    for (int q = 0; q < PF; ++q) {
      const int p = lane + 32 * q;
      if (p < npairs) {
        const int ij = pair_ij[p];
        const int i = ij >> 8, j = ij & 255;
        S[i * SS + j] = gpre[q];
        S[j * SS + i] = gpre[q];
      }
    }
    for (int p = lane + 32 * PF; p < npairs; p += 32) {
      const float v = __ldg(g + D + p);
      const int ij = pair_ij[p];
      const int i = ij >> 8, j = ij & 255;
      S[i * SS + j] = v;
      S[j * SS + i] = v;
    }
    const float4 g0 = g0pre;
    const bool more = b + stride < P.B;
    const float* src[2] = {nullptr, nullptr};
    if (more) {
      prefetch(b + stride);
      dot_resolve_rows<IdT>(P, b + stride, lane, src);  // id loads fly under the FMA loop
    }
    __syncwarp();
    mbar_wait(bar, parity);
    parity ^= 1;
    // one i-tile of 2*RPN rows (RPN = 4 except for the last tile, which only computes the row
    // pairs that exist: 27 rows = 8 + 8 + 8 + 4, not 32).
    // packed fp32x2 FMAs (sm_100 FFMA2), pairing ROWS: acc2[rp][c] = {dX[i0+2rp][d0+c],
    // dX[i0+2rp+1][d0+c]}; the S pairs come straight out of the 128-bit loads and only the 4
    // x values are duplicated in registers (a duplicated {s,s} tile in shared memory was
    // measured slower: two warps of occupancy and twice the shared loads)
    auto tile = [&](auto rpn_tag, int i0, int d0) {
      constexpr int RPN = decltype(rpn_tag)::value;
      float2 acc2[RPN][4];
#pragma unroll
      for (int rp = 0; rp < RPN; ++rp)
#pragma unroll
        for (int c = 0; c < 4; ++c) acc2[rp][c] = make_float2(0.f, 0.f);
#pragma unroll (CF1 ? CF1 : 3)
      for (int j = 0; j < F1; ++j) {
        const float4 xj = *reinterpret_cast<const float4*>(xt + j * RS + d0);
        const float4 s0 = *reinterpret_cast<const float4*>(S + j * SS + i0);
        float4 s1 = make_float4(0.f, 0.f, 0.f, 0.f);
        if (RPN > 2) s1 = *reinterpret_cast<const float4*>(S + j * SS + i0 + 4);
        const float2 sp[4] = {make_float2(s0.x, s0.y), make_float2(s0.z, s0.w),
                              make_float2(s1.x, s1.y), make_float2(s1.z, s1.w)};
        const float2 xx[4] = {make_float2(xj.x, xj.x), make_float2(xj.y, xj.y),
                              make_float2(xj.z, xj.z), make_float2(xj.w, xj.w)};
#pragma unroll
        for (int rp = 0; rp < RPN; ++rp)
#pragma unroll
          for (int c = 0; c < 4; ++c) acc2[rp][c] = __ffma2_rn(sp[rp], xx[c], acc2[rp][c]);
      }
#pragma unroll
      for (int r = 0; r < 2 * RPN; ++r) {
        const int i = i0 + r;
        if (i < F1) {
          const int rp = r >> 1;
          float4 v = (r & 1) ? make_float4(acc2[rp][0].y, acc2[rp][1].y, acc2[rp][2].y, acc2[rp][3].y)
                             : make_float4(acc2[rp][0].x, acc2[rp][1].x, acc2[rp][2].x, acc2[rp][3].x);
          float* dst;
          if (P.peer_gptr && i > 0) {  // straight into the owner's gradient buffer over NVLink
            const long long id = (long long)ids_w[i - 1];
            int gq = 0;
            long long row;
            if (id >= 0) peer_split(P, i - 1, id, gq, row);
            const int e = (i - 1) * P.peer_G + gq;
            dst = reinterpret_cast<float*>(P.peer_gptr[e]) + (P.sample0 + b) * P.peer_gstr[e] + d0;
          } else {
            dst = P.gbase[i] + b * P.gstride[i] + d0;
          }
          if (i == 0) {  // out[:, :D] is X[0] itself
            if (d0 == lane * 4) {
              v.x += g0.x; v.y += g0.y; v.z += g0.z; v.w += g0.w;
            } else {       // D > 128: later column passes
              v.x += __ldg(g + d0);
              v.y += __ldg(g + d0 + 1);
              v.z += __ldg(g + d0 + 2);
              v.w += __ldg(g + d0 + 3);
            }
          }
          *reinterpret_cast<float4*>(dst) = v;
        }
      }
    };
    for (int d0 = lane * 4; d0 < D; d0 += 128) {
      if constexpr (CF1 > 0) {     // the tiles and their row-pair counts are known: straight-line code
        static_assert(CF1 <= 32, "compile-time row count: at most four 8-row tiles");
        constexpr int NT = (CF1 + 7) / 8;
        tile(std::integral_constant<int, bwd_tile_rpn(CF1, 0)>{}, 0, d0);
        if constexpr (NT > 1) tile(std::integral_constant<int, bwd_tile_rpn(CF1, 1)>{}, 8, d0);
        if constexpr (NT > 2) tile(std::integral_constant<int, bwd_tile_rpn(CF1, 2)>{}, 16, d0);
        if constexpr (NT > 3) tile(std::integral_constant<int, bwd_tile_rpn(CF1, 3)>{}, 24, d0);
      } else {
        for (int i0 = 0; i0 < F1; i0 += 8) {
          const int left = F1 - i0;
          if (left > 6) tile(std::integral_constant<int, 4>{}, i0, d0);
          else if (left > 4) tile(std::integral_constant<int, 3>{}, i0, d0);
          else if (left > 2) tile(std::integral_constant<int, 2>{}, i0, d0);
          else tile(std::integral_constant<int, 1>{}, i0, d0);
        }
      }
    }
    __syncwarp();
    if (more) dot_issue_resolved(P, xt, RS, bar, lane, src);
  }
}

static int dot_check_common(long long B, int F1, int D) {
  if (B < 0 || F1 < 2 || D <= 0) return RTF_E_ARG;
  if (F1 > RTF_MAX_FIELDS || D % 4 || D > 1024) return RTF_E_RANGE;
  return 0;
}

template <typename Kern>
static int dot_launch(Kern kern, const DotParams& P, int warp_floats, int cta_floats,
                      cudaStream_t st, int max_warps = 16) {
  const size_t max_smem = 227 * 1024;
  const size_t per_warp = (size_t)warp_floats * 4;
  int nwarps = (int)((max_smem - (size_t)cta_floats * 4) / per_warp);
  if (nwarps < 1) return RTF_E_RANGE;
  if (nwarps > max_warps) nwarps = max_warps;
  const size_t smem = (size_t)cta_floats * 4 + per_warp * nwarps;
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return (int)e;
  long long blocks = (P.B + nwarps - 1) / nwarps;
  if (blocks > kNumSMs) blocks = kNumSMs;  // persistent: one CTA per SM
  kern<<<(unsigned)blocks, nwarps * 32, smem, st>>>(P, warp_floats);
  RTF_CHECK_LAUNCH();
  return 0;
}

static int dot_fwd_impl(DotParams& P, int ids_i64, cudaStream_t st) {
  const int F1p = (P.F1 + 3) & ~3, RS = dot_row_stride(P.D);
  const int npairs = P.F1 * (P.F1 - 1) / 2;
  // 7x7 register blocks (instantiated for the shape the bench and the reference's Criteo DLRM
  // use; every other shape takes the generic 4x4 kernel)
  if ((P.F1 + 6) / 7 == 4 && P.D == 128) {     // the Criteo shape: 22..28 rows of 128
    const int wf = 28 * RS + ((28 * 29 + 3) & ~3) + 4;    // rows, Z tile, mbarrier
    const int cf = ((npairs + 1) / 2 + 3) & ~3;           // pair table
    // 12 warps (154 registers each); measured 12 / 11 / 10 / 8 warps: 0.305 / 0.327 / 0.374 / 0.396 ms
    return ids_i64 ? dot_launch(dot_fwd7_kernel<int64_t, 128, 4>, P, wf, cf, st, 12)
                   : dot_launch(dot_fwd7_kernel<int32_t, 128, 4>, P, wf, cf, st, 12);
  }
  const int warp_floats = F1p * RS + ((npairs + 3) & ~3) + 4;  // + mbarrier (8 B, 16-B slot)
  return ids_i64 ? dot_launch(dot_fwd_kernel<int64_t>, P, warp_floats, 0, st)
                 : dot_launch(dot_fwd_kernel<int32_t>, P, warp_floats, 0, st);
}
static int dot_bwd_impl(DotParams& P, int ids_i64, cudaStream_t st) {
  const int F1p = (P.F1 + 7) & ~7, RS = dot_row_stride(P.D);
  const int npairs = P.F1 * (P.F1 - 1) / 2;
  const int warp_floats = P.F1 * RS + P.F1 * (F1p + 4) + 4 + 128;  // + mbarrier slot + 64 ids
  const int cta_floats = ((npairs + 1) / 2 + 3) & ~3;
  if (P.F1 == 27 && P.D == 128)    // the Criteo shape (26 tables + the dense row)
    return ids_i64 ? dot_launch(dot_bwd_kernel<int64_t, 27, 128>, P, warp_floats, cta_floats, st, 12)
                   : dot_launch(dot_bwd_kernel<int32_t, 27, 128>, P, warp_floats, cta_floats, st, 12);
  return ids_i64 ? dot_launch(dot_bwd_kernel<int64_t>, P, warp_floats, cta_floats, st)
                 : dot_launch(dot_bwd_kernel<int32_t>, P, warp_floats, cta_floats, st);
}

static int dot_fill_tables(DotParams& P, const float* const* tables, const int64_t* rows,
                           int n_fields) {
  for (int f = 0; f < n_fields; ++f) {
    if (!tables[f] || rows[f] <= 0) return RTF_E_ARG;
    if ((uintptr_t)tables[f] % 16) return RTF_E_ALIGN;
    P.table[f] = tables[f];
    P.rows[f] = rows[f];
  }
  return 0;
}

}  // namespace rtf

using namespace rtf;

static void dot_rows_stacked(DotParams& P, const float* x, float* gx, int F1, int D) {
  for (int i = 0; i < F1; ++i) {
    P.rbase[i] = x + (long long)i * D;
    P.rstride[i] = (long long)F1 * D;
    P.gbase[i] = gx ? gx + (long long)i * D : nullptr;
    P.gstride[i] = (long long)F1 * D;
  }
}

extern "C" int rtf_dot_interact_fwd(const float* d_x, int64_t B, int F1, int D, float* d_out,
                                    int64_t out_sb, int out_cols, void* stream) {
  int rc = dot_check_common(B, F1, D);
  if (rc) return rc;
  if (B == 0) return 0;
  if (!d_x || !d_out) return RTF_E_ARG;
  const int need = D + F1 * (F1 - 1) / 2;
  if (out_cols < need || out_sb < out_cols) return RTF_E_ARG;
  if ((uintptr_t)d_x % 16) return RTF_E_ALIGN;
  DotParams P = {};
  dot_rows_stacked(P, d_x, nullptr, F1, D);
  P.B = B; P.F1 = F1; P.D = D; P.out = d_out; P.out_sb = out_sb; P.out_cols = out_cols;
  return dot_fwd_impl(P, 0, (cudaStream_t)stream);
}

extern "C" int rtf_dot_interact_bwd(const float* d_x, const float* d_gout, int64_t gout_sb,
                                    int64_t B, int F1, int D, float* d_gx, void* stream) {
  int rc = dot_check_common(B, F1, D);
  if (rc) return rc;
  if (B == 0) return 0;
  if (!d_x || !d_gout || !d_gx) return RTF_E_ARG;
  if (gout_sb < D + F1 * (F1 - 1) / 2) return RTF_E_ARG;
  if ((uintptr_t)d_x % 16 || (uintptr_t)d_gx % 16) return RTF_E_ALIGN;
  DotParams P = {};
  dot_rows_stacked(P, d_x, d_gx, F1, D);
  P.B = B; P.F1 = F1; P.D = D; P.gout = d_gout; P.gout_sb = gout_sb;
  return dot_bwd_impl(P, 0, (cudaStream_t)stream);
}

// rows given one by one: row i of sample b at row_base[i] + b*row_stride[i] (HOST arrays of F1
// device pointers / element strides).  This is how the sharded path interacts straight out of
// the all-to-all receive buffer (source-major blocks) without a permute copy.
extern "C" int rtf_dot_rows_fwd(const float* const* row_base, const int64_t* row_stride, int F1,
                                int D, int64_t B, float* d_out, int64_t out_sb, int out_cols,
                                float* d_xsave, int64_t xsave_sb, void* stream) {
  int rc = dot_check_common(B, F1, D);
  if (rc) return rc;
  if (B == 0) return 0;
  if (!row_base || !row_stride || !d_out) return RTF_E_ARG;
  const int need = D + F1 * (F1 - 1) / 2;
  if (out_cols < need || out_sb < out_cols) return RTF_E_ARG;
  DotParams P = {};
  for (int i = 0; i < F1; ++i) {
    if (!row_base[i]) return RTF_E_ARG;
    if ((uintptr_t)row_base[i] % 16 || row_stride[i] % 4) return RTF_E_ALIGN;
    P.rbase[i] = row_base[i];
    P.rstride[i] = row_stride[i];
  }
  if (d_xsave && ((uintptr_t)d_xsave % 16 || xsave_sb % 4 || xsave_sb < (int64_t)(F1 - 1) * D))
    return RTF_E_ALIGN;
  P.xsave = d_xsave; P.xsave_sb = xsave_sb;
  P.B = B; P.F1 = F1; P.D = D; P.out = d_out; P.out_sb = out_sb; P.out_cols = out_cols;
  return dot_fwd_impl(P, 0, (cudaStream_t)stream);
}

extern "C" int rtf_dot_rows_bwd(const float* const* row_base, const int64_t* row_stride, int F1,
                                int D, int64_t B, const float* d_gout, int64_t gout_sb,
                                float* const* grad_base, const int64_t* grad_stride,
                                void* stream) {
  int rc = dot_check_common(B, F1, D);
  if (rc) return rc;
  if (B == 0) return 0;
  if (!row_base || !row_stride || !d_gout || !grad_base || !grad_stride) return RTF_E_ARG;
  if (gout_sb < D + F1 * (F1 - 1) / 2) return RTF_E_ARG;
  DotParams P = {};
  for (int i = 0; i < F1; ++i) {
    if (!row_base[i] || !grad_base[i]) return RTF_E_ARG;
    if ((uintptr_t)row_base[i] % 16 || row_stride[i] % 4 || (uintptr_t)grad_base[i] % 16 ||
        grad_stride[i] % 4)
      return RTF_E_ALIGN;
    P.rbase[i] = row_base[i];
    P.rstride[i] = row_stride[i];
    P.gbase[i] = grad_base[i];
    P.gstride[i] = grad_stride[i];
  }
  P.B = B; P.F1 = F1; P.D = D; P.gout = d_gout; P.gout_sb = gout_sb;
  return dot_bwd_impl(P, 0, (cudaStream_t)stream);
}

extern "C" int rtf_embed_dot_fwd(const float* const* tables, const int64_t* rows, int n_fields,
                                 int D, const void* d_ids, int ids_i64, int64_t B, int64_t ids_sb,
                                 int64_t ids_sf, const float* d_dense, int64_t dense_sb,
                                 float* d_out, int64_t out_sb, int out_cols, int32_t* d_err,
                                 void* stream) {
  if (!tables || !rows || n_fields < 1) return RTF_E_ARG;
  const int F1 = n_fields + 1;
  int rc = dot_check_common(B, F1, D);
  if (rc) return rc;
  if (B == 0) return 0;
  if (!d_ids || !d_dense || !d_out) return RTF_E_ARG;
  const int need = D + F1 * (F1 - 1) / 2;
  if (out_cols < need || out_sb < out_cols) return RTF_E_ARG;
  if ((uintptr_t)d_dense % 16 || dense_sb % 4) return RTF_E_ALIGN;
  DotParams P = {};
  rc = dot_fill_tables(P, tables, rows, n_fields);
  if (rc) return rc;
  P.gather = 1; P.ids = d_ids; P.ids_sb = ids_sb; P.ids_sf = ids_sf; P.rbase[0] = d_dense;
  P.rstride[0] = dense_sb;
  P.B = B; P.F1 = F1; P.D = D; P.out = d_out; P.out_sb = out_sb; P.out_cols = out_cols;
  P.err = d_err;
  return dot_fwd_impl(P, ids_i64, (cudaStream_t)stream);
}

extern "C" int rtf_embed_dot_bwd(const float* const* tables, const int64_t* rows, int n_fields,
                                 int D, const void* d_ids, int ids_i64, int64_t B, int64_t ids_sb,
                                 int64_t ids_sf, const float* d_dense, int64_t dense_sb,
                                 const float* d_gout, int64_t gout_sb, float* d_gdense,
                                 int64_t gdense_sb, float* d_gemb, int64_t gemb_sb, void* stream) {
  if (!tables || !rows || n_fields < 1) return RTF_E_ARG;
  const int F1 = n_fields + 1;
  int rc = dot_check_common(B, F1, D);
  if (rc) return rc;
  if (B == 0) return 0;
  if (!d_ids || !d_dense || !d_gout || !d_gdense || !d_gemb) return RTF_E_ARG;
  if (gout_sb < D + F1 * (F1 - 1) / 2 || gemb_sb < (int64_t)n_fields * D) return RTF_E_ARG;
  if ((uintptr_t)d_dense % 16 || dense_sb % 4 || (uintptr_t)d_gdense % 16 || gdense_sb % 4 ||
      (uintptr_t)d_gemb % 16 || gemb_sb % 4)
    return RTF_E_ALIGN;
  DotParams P = {};
  rc = dot_fill_tables(P, tables, rows, n_fields);
  if (rc) return rc;
  P.gather = 1; P.ids = d_ids; P.ids_sb = ids_sb; P.ids_sf = ids_sf; P.rbase[0] = d_dense;
  P.rstride[0] = dense_sb;
  P.gbase[0] = d_gdense; P.gstride[0] = gdense_sb;
  for (int f = 0; f < n_fields; ++f) {
    P.gbase[1 + f] = d_gemb + (long long)f * D;
    P.gstride[1 + f] = gemb_sb;
  }
  P.B = B; P.F1 = F1; P.D = D; P.gout = d_gout; P.gout_sb = gout_sb;
  return dot_bwd_impl(P, ids_i64, (cudaStream_t)stream);
}

// ---- tables sharded over G GPUs, rows pulled / gradients pushed through NVLink peer pointers --
// d_peer_tab: device array [n_fields][G] of table-shard base pointers (as int64); a field whose
// bit is set in rw_mask is row-wise sharded (row r on rank r % G at local row r / G), any other
// field lives wholly on one rank whose pointer is entry [f][0].  rows[] (HOST) are the GLOBAL
// row counts (bounds check).  d_xsave keeps the gathered rows for the backward.
// d_peer_str != NULL: the holders already gathered their rows for the global batch (K1) into
// (B_global, T_g*D) buffers; d_peer_tab[f][g] is then the base of field f's column in rank g's
// buffer, d_peer_str[f][g] its sample stride (elements), and the row of local sample b is read
// at sample index sample0 + b — sequential addresses, which NVLink moves 2.2x faster than the
// random table rows (measured at 8 GPUs, DESIGN.md §5).
extern "C" int rtf_embed_dot_peer_fwd(const int64_t* d_peer_tab, const int64_t* d_peer_str,
                                      int64_t sample0, int G, uint64_t rw_mask,
                                      const int64_t* rows, int n_fields, int D, const void* d_ids,
                                      int ids_i64, int64_t B, int64_t ids_sb, int64_t ids_sf,
                                      const float* d_dense, int64_t dense_sb, float* d_out,
                                      int64_t out_sb, int out_cols, float* d_xsave,
                                      int64_t xsave_sb, int32_t* d_err, void* stream) {
  if (!d_peer_tab || !rows || n_fields < 1 || G < 1) return RTF_E_ARG;
  const int F1 = n_fields + 1;
  int rc = dot_check_common(B, F1, D);
  if (rc) return rc;
  if (B == 0) return 0;
  if (!d_ids || !d_dense || !d_out) return RTF_E_ARG;
  const int need = D + F1 * (F1 - 1) / 2;
  if (out_cols < need || out_sb < out_cols) return RTF_E_ARG;
  if ((uintptr_t)d_dense % 16 || dense_sb % 4) return RTF_E_ALIGN;
  if (d_xsave && ((uintptr_t)d_xsave % 16 || xsave_sb % 4 || xsave_sb < (int64_t)n_fields * D))
    return RTF_E_ALIGN;
  DotParams P = {};
  for (int f = 0; f < n_fields; ++f) {
    if (rows[f] <= 0) return RTF_E_ARG;
    P.rows[f] = rows[f];
  }
  P.gather = 1; P.ids = d_ids; P.ids_sb = ids_sb; P.ids_sf = ids_sf; P.rbase[0] = d_dense;
  P.rstride[0] = dense_sb; P.peer_tab = (const long long*)d_peer_tab; P.peer_G = G;
  P.peer_str = (const long long*)d_peer_str; P.sample0 = sample0;
  P.rw_mask = rw_mask; P.xsave = d_xsave; P.xsave_sb = xsave_sb;
  P.B = B; P.F1 = F1; P.D = D; P.out = d_out; P.out_sb = out_sb; P.out_cols = out_cols;
  P.err = d_err;
  return dot_fwd_impl(P, ids_i64, (cudaStream_t)stream);
}

// backward of the above: X rows come from d_xsave (local), dX row of field f goes to
// d_peer_gptr[f][g] + (sample0 + b) * d_peer_gstr[f][g] with g = id % G for row-wise fields, 0
// otherwise — i.e. straight into the owning rank's gradient buffer (K2's d_grad there).
extern "C" int rtf_embed_dot_peer_bwd(const float* d_xsave, int64_t xsave_sb, const int64_t* rows,
                                      int n_fields, int D, const void* d_ids, int ids_i64,
                                      int64_t B, int64_t ids_sb, int64_t ids_sf,
                                      const float* d_dense, int64_t dense_sb, const float* d_gout,
                                      int64_t gout_sb, float* d_gdense, int64_t gdense_sb,
                                      const int64_t* d_peer_gptr, const int64_t* d_peer_gstr, int G,
                                      uint64_t rw_mask, int64_t sample0, void* stream) {
  if (!d_peer_gptr || !d_peer_gstr || !rows || n_fields < 1 || G < 1) return RTF_E_ARG;
  const int F1 = n_fields + 1;
  int rc = dot_check_common(B, F1, D);
  if (rc) return rc;
  if (B == 0) return 0;
  if (!d_xsave || !d_ids || !d_dense || !d_gout || !d_gdense) return RTF_E_ARG;
  if (gout_sb < D + F1 * (F1 - 1) / 2) return RTF_E_ARG;
  if ((uintptr_t)d_dense % 16 || dense_sb % 4 || (uintptr_t)d_gdense % 16 || gdense_sb % 4 ||
      (uintptr_t)d_xsave % 16 || xsave_sb % 4)
    return RTF_E_ALIGN;
  DotParams P = {};
  for (int f = 0; f < n_fields; ++f) {
    P.rows[f] = rows[f];
    P.rbase[1 + f] = d_xsave + (long long)f * D;
    P.rstride[1 + f] = xsave_sb;
  }
  P.rbase[0] = d_dense; P.rstride[0] = dense_sb;
  P.gbase[0] = d_gdense; P.gstride[0] = gdense_sb;
  P.ids = d_ids; P.ids_sb = ids_sb; P.ids_sf = ids_sf;
  P.peer_gptr = (const long long*)d_peer_gptr; P.peer_gstr = (const long long*)d_peer_gstr;
  P.peer_G = G; P.rw_mask = rw_mask; P.sample0 = sample0;
  P.B = B; P.F1 = F1; P.D = D; P.gout = d_gout; P.gout_sb = gout_sb;
  return dot_bwd_impl(P, ids_i64, (cudaStream_t)stream);
}
