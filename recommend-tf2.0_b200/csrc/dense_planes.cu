// fp32 -> three bf16 planes for the plane-fed dense GEMM (dense_gemm_planes.cuh).
//
// planes[p * plane_stride + r * ld_out + c] = plane p of x[r * ld_in + c] (rtf::split_bf16x3), for
// r < rows, c < cols: 4 B read and 6 B written per value.  Contiguous rows (ld_in == ld_out ==
// cols, cols % 4 == 0, the layout core.split_planes makes) take a flat pass with no index
// arithmetic: 16-byte loads and three 8-byte stores per thread, two quads in flight.  Other
// layouts split one pair of columns per thread (8-byte load, three 4-byte stores).
#include "rtf_common.cuh"

namespace rtf {

__global__ void __launch_bounds__(256)
split_bf16x3_kernel(const float* __restrict__ x, long long rows, int cols, long long ld_in,
                    uint32_t* __restrict__ planes, long long ld_out, long long plane_stride) {
  const int pr = cols / 2;  // pairs per row
  const long long n = rows * pr;
  const long long ps = plane_stride / 2;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n;
       i += (long long)gridDim.x * blockDim.x) {
    const long long r = i / pr;
    const int c = (int)(i - r * pr) * 2;
    const float2 v = *reinterpret_cast<const float2*>(x + r * ld_in + c);
    uint32_t p0, p1, p2;
    split_bf16x3(v.x, v.y, p0, p1, p2);
    uint32_t* dst = planes + (r * ld_out + c) / 2;
    dst[0] = p0;
    dst[ps] = p1;
    dst[2 * ps] = p2;
  }
}

__global__ void __launch_bounds__(256)
split_bf16x3_flat_kernel(const float4* __restrict__ x, long long n4, uint2* __restrict__ planes,
                         long long ps4) {
  const long long stride = (long long)gridDim.x * blockDim.x;
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  for (; i + stride < n4; i += 2 * stride) {
    const float4 a = ldg_nc_f4(reinterpret_cast<const float*>(x + i));
    const float4 b = ldg_nc_f4(reinterpret_cast<const float*>(x + i + stride));
    uint2 a0, a1, a2, b0, b1, b2;
    split_bf16x3(a.x, a.y, a0.x, a1.x, a2.x);
    split_bf16x3(a.z, a.w, a0.y, a1.y, a2.y);
    split_bf16x3(b.x, b.y, b0.x, b1.x, b2.x);
    split_bf16x3(b.z, b.w, b0.y, b1.y, b2.y);
    planes[i] = a0;
    planes[i + ps4] = a1;
    planes[i + 2 * ps4] = a2;
    planes[i + stride] = b0;
    planes[i + stride + ps4] = b1;
    planes[i + stride + 2 * ps4] = b2;
  }
  if (i < n4) {
    const float4 a = ldg_nc_f4(reinterpret_cast<const float*>(x + i));
    uint2 a0, a1, a2;
    split_bf16x3(a.x, a.y, a0.x, a1.x, a2.x);
    split_bf16x3(a.z, a.w, a0.y, a1.y, a2.y);
    planes[i] = a0;
    planes[i + ps4] = a1;
    planes[i + 2 * ps4] = a2;
  }
}

}  // namespace rtf

extern "C" int rtf_split_bf16x3(const float* d_x, int64_t rows, int cols, int64_t ld_in,
                                uint16_t* d_planes, int64_t ld_out, int64_t plane_stride,
                                void* stream) {
  if (!d_x || !d_planes || rows < 0 || cols < 0) return RTF_E_ARG;
  if (cols % 2 || ld_in % 2 || ld_out % 2 || plane_stride % 2 || ld_in < cols || ld_out < cols ||
      plane_stride < rows * ld_out || (uintptr_t)d_x % 8 || (uintptr_t)d_planes % 4)
    return RTF_E_ALIGN;
  if (rows == 0 || cols == 0) return 0;
  if (ld_in == cols && ld_out == cols && cols % 4 == 0 && plane_stride % 4 == 0 &&
      (uintptr_t)d_x % 16 == 0 && (uintptr_t)d_planes % 8 == 0) {
    const long long n4 = rows * cols / 4;
    const int grid = (int)std::min<long long>((n4 + 511) / 512, (long long)rtf::kNumSMs * 16);
    rtf::split_bf16x3_flat_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(
        reinterpret_cast<const float4*>(d_x), n4, reinterpret_cast<uint2*>(d_planes),
        plane_stride / 4);
    RTF_CHECK_LAUNCH();
    return 0;
  }
  const long long work = rows * (cols / 2);
  const int grid = (int)std::min<long long>((work + 255) / 256, (long long)rtf::kNumSMs * 32);
  rtf::split_bf16x3_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(
      d_x, rows, cols, ld_in, reinterpret_cast<uint32_t*>(d_planes), ld_out, plane_stride);
  RTF_CHECK_LAUNCH();
  return 0;
}
