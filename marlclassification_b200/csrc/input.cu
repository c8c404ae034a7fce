// Device side of the input pipeline (SURVEY.md 8(f) rank 3).
//
// The reference decodes images with PIL (uint8, H x W x C) and converts them on the host with
// torchvision's ToTensor (registry.py:56-57): permute to C x H x W, cast to fp32, divide by 255.
// Here the uint8 pixels go over PCIe as they are (4x fewer bytes than fp32) and one HBM-bound
// kernel does permute + cast + divide: 1 byte read and 4 bytes written per element.  The result is
// bit-identical to ToTensor: (float)u / 255.0f is the same IEEE division.
#include <stdlib.h>

#include <algorithm>

#include "common.cuh"

namespace marlc {

// HWC uint8 -> CHW fp32, one image ROW per threadIdx.y (needs W % 4 == 0 so the 4*C source bytes of
// 4 pixels start on a 4-byte boundary): the row's (b, y) is one 32-bit division per thread and the
// position inside the row needs none.  A 1-D grid over groups of 4 pixels pays two 64-bit divisions
// (~200 instructions) per 4 pixels, more issue time than the 60 bytes they move cost in HBM time
// (A/B in profiles/README.md).
template <int C>
__global__ void __launch_bounds__(256) u8hwc_to_f32chw_rows_kernel(const uint8_t* __restrict__ src,
                                                                   float* __restrict__ dst, int rows, int H, int W) {
    const int w4 = W >> 2;
    for (int row = blockIdx.x * blockDim.y + threadIdx.y; row < rows; row += gridDim.x * blockDim.y) {
        const int b = row / H, y = row - b * H;
        const uint32_t* s_row = reinterpret_cast<const uint32_t*>(src + (long)row * W * C);
        float* d_row = dst + ((long)b * C * H + y) * W;
        for (int x4 = threadIdx.x; x4 < w4; x4 += blockDim.x) {
            uint32_t wds[C];
#pragma unroll
            for (int i = 0; i < C; ++i) wds[i] = __ldg(s_row + x4 * C + i);
            float px[4 * C];
#pragma unroll
            for (int i = 0; i < 4 * C; ++i) px[i] = (float)((wds[i >> 2] >> (8 * (i & 3))) & 0xFFu) / 255.0f;
#pragma unroll
            for (int c = 0; c < C; ++c)
                __stcs(reinterpret_cast<float4*>(d_row + (long)c * H * W + 4 * x4),
                       make_float4(px[c], px[C + c], px[2 * C + c], px[3 * C + c]));
        }
    }
}

// generic fallback (any C, any W): one thread per output element, coalesced writes
__global__ void __launch_bounds__(256) u8hwc_to_f32chw_generic_kernel(const uint8_t* __restrict__ src,
                                                                      float* __restrict__ dst, long total, int C, int H,
                                                                      int W) {
    for (long e = blockIdx.x * (long)blockDim.x + threadIdx.x; e < total; e += (long)gridDim.x * blockDim.x) {
        const int x = (int)(e % W);
        long r = e / W;
        const int y = (int)(r % H);
        r /= H;
        const int c = (int)(r % C);
        const long b = r / C;
        dst[e] = (float)__ldg(src + ((b * H + y) * (long)W + x) * C + c) / 255.0f;
    }
}

// same layout on both sides (CHW uint8, e.g. torchvision.io.decode_*): cast + divide only
__global__ void __launch_bounds__(256) u8_to_f32_kernel(const uint8_t* __restrict__ src, float* __restrict__ dst, long n) {
    const long n16 = n >> 4;
    const uint4* s16 = reinterpret_cast<const uint4*>(src);
    for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < n16; i += (long)gridDim.x * blockDim.x) {
        const uint4 v = __ldg(s16 + i);
        const uint32_t w[4] = {v.x, v.y, v.z, v.w};
        float4* d = reinterpret_cast<float4*>(dst + (i << 4));
#pragma unroll
        for (int q = 0; q < 4; ++q)
            __stcs(d + q, make_float4((float)(w[q] & 0xFFu) / 255.0f, (float)((w[q] >> 8) & 0xFFu) / 255.0f,
                                      (float)((w[q] >> 16) & 0xFFu) / 255.0f, (float)(w[q] >> 24) / 255.0f));
    }
    for (long i = (n16 << 4) + blockIdx.x * (long)blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x)
        dst[i] = (float)src[i] / 255.0f;
}

template <int C>
static void launch_rows(const uint8_t* src, float* dst, int rows, int H, int W, cudaStream_t s) {
    const int w4 = W >> 2;
    const int tx = std::min(256, (w4 + 31) & ~31), ty = std::max(1, 256 / tx);
    const long blocks = ((long)rows + ty - 1) / ty;
    const int grid = (int)std::max(1L, std::min(blocks, 148L * 32));
    u8hwc_to_f32chw_rows_kernel<C><<<grid, dim3(tx, ty), 0, s>>>(src, dst, rows, H, W);
}

static int grid_for(long work_items) {
    const long blocks = (work_items + 255) / 256;
    return (int)std::max(1L, std::min(blocks, 148L * 16));  // grid-stride beyond 16 CTAs per SM
}

}  // namespace marlc

using namespace marlc;

extern "C" int marlc_images_u8_to_f32(const uint8_t* src, float* dst, int B, int C, int H, int W, int src_hwc,
                                      void* stream) {
    MARLC_CHECK(src && dst, "images_u8_to_f32: null buffer");
    MARLC_CHECK(B >= 0 && C >= 1 && H >= 1 && W >= 1, "images_u8_to_f32: bad shape B=%d C=%d H=%d W=%d", B, C, H, W);
    cudaStream_t s = (cudaStream_t)stream;
    const long total = (long)B * C * H * W;
    if (total == 0) return 0;
    if (!src_hwc || C == 1) {
        const bool al = (((uintptr_t)src & 15) == 0) && (((uintptr_t)dst & 15) == 0);
        if (al) u8_to_f32_kernel<<<grid_for(total >> 4), 256, 0, s>>>(src, dst, total);
        else u8hwc_to_f32chw_generic_kernel<<<grid_for(total), 256, 0, s>>>(src, dst, total, 1, 1, 1024);  // identity order
    } else {
        const bool vec = (W % 4 == 0) && (((uintptr_t)src & 3) == 0) && (((uintptr_t)dst & 15) == 0);
        const bool rows = vec && (long)B * H < 0x7fffffffL;
        if (rows && C == 3) launch_rows<3>(src, dst, B * H, H, W, s);
        else if (rows && C == 4) launch_rows<4>(src, dst, B * H, H, W, s);
        else if (rows && C == 2) launch_rows<2>(src, dst, B * H, H, W, s);
        else u8hwc_to_f32chw_generic_kernel<<<grid_for(total), 256, 0, s>>>(src, dst, total, C, H, W);
    }
    MARLC_LAUNCH_CHECK();
    return 0;
}
