// First convolution of the network (down1.net.0, unet_model.py:29 -> :10-12):
// Conv2d(n_channels -> 64, 3x3, pad 1) + folded BatchNorm + ReLU.
//
// K = 9 * n_channels = 27 is far too thin for the tensor cores and the layer is
// HBM-bound (it writes 64 bf16 channels per pixel, reads 3 floats): it runs on
// the CUDA cores in fp32 and doubles as the ingest stage -- it reads the user's
// tensor as it is (fp32 NCHW like inference.py:36-42 produces, or the raw uint8
// HWC frame, scaled by /255 here) and writes the NHWC bf16 layout every later
// kernel consumes.
//
// Float inputs may also be fp16 / bf16 and NCHW or NHWC (the storage of a channels_last tensor): an element is
// widened to fp32 where it is read, which is exact for every 16-bit value, so everything after the read sees the
// same fp32 value as for the fp32 NCHW tensor x.float().contiguous().
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include "ptx.cuh"

namespace ub {

// input formats (include/unetb200.h UNETB200_X_*); NHWC = [N][H][W][C] in memory
enum : int { X_F32_NCHW = 0, X_U8_NHWC = 1, X_F16_NCHW = 2, X_BF16_NCHW = 3, X_F32_NHWC = 4, X_F16_NHWC = 5,
             X_BF16_NHWC = 6 };
// kernel template argument "format chosen at run time": X_F32_NCHW or X_U8_NHWC by the launch's x_fmt / stem_fmt
// (the two original formats share one instantiation per kernel; every other format has its own)
constexpr int X_RUNTIME = -1;
constexpr int kNumXFormats = 7;

__host__ __device__ constexpr int x_elem_bytes(int f) {
    return f == X_U8_NHWC ? 1 : ((f == X_F32_NCHW || f == X_F32_NHWC) ? 4 : 2);
}
__host__ __device__ constexpr bool x_is_nhwc(int f) { return f == X_U8_NHWC || f >= X_F32_NHWC; }
__host__ __device__ constexpr int x_per_16B(int f) { return 16 / x_elem_bytes(f); }

// Input box of the tensor-core stem (conv_tc.cuh A_STEM, make_input_map): the 18 x 10 halo patch of a tile is one
// TMA box, and a TMA tile load faults unless the byte offset of its innermost start coordinate is a multiple of 16.
//   NCHW: 4-D map (W, H, C, N), box (stem_box_w, 18, C, 1) from column x0 - (x_per_16B - 1): patch columns
//         x_per_16B - 1 .. x_per_16B + 8 of the box rows
//   NHWC: 3-D map (W * C, H, N), box (stem_box_w, 18, 1) from the 16-byte floor of x0 * C: the patch starts
//         sh = (x0 * C) mod x_per_16B elements into each box row
// with x0 = the tile's first column - 1.  The width is the smallest 16-byte multiple that covers the patch row
// from any start: fp32 NCHW 16, 16-bit NCHW 24, NHWC (C = 3) fp32 36 / 16-bit 40 / uint8 48 elements.
__host__ __device__ constexpr int stem_box_w(int f, int cin) {
    return ((x_is_nhwc(f) ? 10 * cin : 10) + 2 * (x_per_16B(f) - 1)) / x_per_16B(f) * x_per_16B(f);
}
__host__ __device__ constexpr int stem_box_bytes(int f, int cin) {
    return stem_box_w(f, cin) * x_elem_bytes(f) * 18 * (x_is_nhwc(f) ? 1 : cin);
}

// 16-bit element -> fp32 (exact)
template <int XF>
__device__ __forceinline__ float x_widen16(uint16_t u) {
    if constexpr (XF == X_F16_NCHW || XF == X_F16_NHWC) return __half2float(__ushort_as_half(u));
    else return __uint_as_float(static_cast<uint32_t>(u) << 16);
}

// element i of a float-format input in global memory, as fp32
template <int XF>
__device__ __forceinline__ float x_load(const void* x, size_t i) {
    static_assert(XF != X_U8_NHWC && XF != X_RUNTIME, "float formats only");
    if constexpr (x_elem_bytes(XF) == 4) return __ldg(static_cast<const float*>(x) + i);
    else return x_widen16<XF>(__ldg(static_cast<const unsigned short*>(x) + i));
}

struct StemParams {
    const void* x;        // input, format per x_fmt
    const float* w;       // [9*CIN][64] fp32, k = (ky*3+kx)*CIN + ci, BN folded
    const float* bias;    // [64]
    void* out;            // [N][H][W][64] bf16
    int N, H, W;
    int x_fmt;
};

constexpr int kStemTX = 32, kStemTY = 8;

template <int CIN, int XF = X_RUNTIME>
__global__ void __launch_bounds__(256) stem_conv_kernel(const StemParams p) {
    __shared__ __align__(16) float s_w[9 * CIN * 64];
    __shared__ __align__(16) float s_b[64];
    __shared__ float s_in[CIN][kStemTY + 2][kStemTX + 2];

    const int n = blockIdx.z;
    const int x0 = blockIdx.x * kStemTX, y0 = blockIdx.y * kStemTY;
    const int tid = threadIdx.x;

    for (int i = tid; i < 9 * CIN * 64; i += 256) s_w[i] = p.w[i];
    if (tid < 64) s_b[tid] = p.bias[tid];
    // halo tile, zero outside the image (= conv zero padding)
    for (int i = tid; i < CIN * (kStemTY + 2) * (kStemTX + 2); i += 256) {
        const int ci = i / ((kStemTY + 2) * (kStemTX + 2));
        const int rem = i - ci * ((kStemTY + 2) * (kStemTX + 2));
        const int yy = rem / (kStemTX + 2), xx = rem - yy * (kStemTX + 2);
        const int y = y0 + yy - 1, x = x0 + xx - 1;
        float v = 0.f;
        if (y >= 0 && y < p.H && x >= 0 && x < p.W) {
            if constexpr (XF != X_RUNTIME) {
                v = x_load<XF>(p.x, x_is_nhwc(XF) ? ((static_cast<size_t>(n) * p.H + y) * p.W + x) * CIN + ci
                                                  : ((static_cast<size_t>(n) * CIN + ci) * p.H + y) * p.W + x);
            } else if (p.x_fmt == X_F32_NCHW) {
                v = __ldg(static_cast<const float*>(p.x) +
                          ((static_cast<size_t>(n) * CIN + ci) * p.H + y) * p.W + x);
            } else {
                const uint8_t u = __ldg(static_cast<const uint8_t*>(p.x) +
                                        ((static_cast<size_t>(n) * p.H + y) * p.W + x) * CIN + ci);
                v = __fdiv_rn(static_cast<float>(u), 255.0f);   // inference.py:36 (`/ 255.0`)
            }
        }
        s_in[ci][yy][xx] = v;
    }
    __syncthreads();

    const int tx = tid & 31, ty = tid >> 5;
    const int x = x0 + tx, y = y0 + ty;
    float v[9 * CIN];
#pragma unroll
    for (int ky = 0; ky < 3; ++ky)
#pragma unroll
        for (int kx = 0; kx < 3; ++kx)
#pragma unroll
            for (int ci = 0; ci < CIN; ++ci) v[(ky * 3 + kx) * CIN + ci] = s_in[ci][ty + ky][tx + kx];

    if (x >= p.W || y >= p.H) return;
    uint4* dst = reinterpret_cast<uint4*>(static_cast<uint16_t*>(p.out) +
                                          ((static_cast<size_t>(n) * p.H + y) * p.W + x) * 64);
#pragma unroll 1
    for (int half = 0; half < 2; ++half) {
        float acc[32];
#pragma unroll
        for (int c = 0; c < 32; ++c) acc[c] = s_b[half * 32 + c];
#pragma unroll
        for (int k = 0; k < 9 * CIN; ++k) {
            const float4* wr = reinterpret_cast<const float4*>(s_w + k * 64 + half * 32);
#pragma unroll
            for (int c4 = 0; c4 < 8; ++c4) {
                const float4 w4 = wr[c4];
                acc[c4 * 4 + 0] = fmaf(v[k], w4.x, acc[c4 * 4 + 0]);
                acc[c4 * 4 + 1] = fmaf(v[k], w4.y, acc[c4 * 4 + 1]);
                acc[c4 * 4 + 2] = fmaf(v[k], w4.z, acc[c4 * 4 + 2]);
                acc[c4 * 4 + 3] = fmaf(v[k], w4.w, acc[c4 * 4 + 3]);
            }
        }
#pragma unroll
        for (int c8 = 0; c8 < 4; ++c8) {
            uint4 o;
            o.x = pack_bf16x2(fmaxf(acc[c8 * 8 + 0], 0.f), fmaxf(acc[c8 * 8 + 1], 0.f));
            o.y = pack_bf16x2(fmaxf(acc[c8 * 8 + 2], 0.f), fmaxf(acc[c8 * 8 + 3], 0.f));
            o.z = pack_bf16x2(fmaxf(acc[c8 * 8 + 4], 0.f), fmaxf(acc[c8 * 8 + 5], 0.f));
            o.w = pack_bf16x2(fmaxf(acc[c8 * 8 + 6], 0.f), fmaxf(acc[c8 * 8 + 7], 0.f));
            dst[half * 4 + c8] = o;
        }
    }
}

}  // namespace ub
