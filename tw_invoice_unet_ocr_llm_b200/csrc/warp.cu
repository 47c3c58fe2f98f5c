// Ragged batch of affine crops (include/unetb200.h, unetb200_warp_crops): every output pixel of every crop is one
// bilinear sample of its source frame, bit-identical to
//   cv2.warpAffine(src, M, (out_w, out_h), flags=INTER_LINEAR | WARP_INVERSE_MAP, borderMode=BORDER_REPLICATE)
// for uint8 RGB frames.  OpenCV's fixed point (imgwarp.cpp, AB_BITS = 10, INTER_BITS = 5):
//   X = (rint((M01 i + M02) * 1024) + 16 + rint((M00 j) * 1024)) >> 5      (Y likewise with M10, M11, M12)
//   integer part X >> 5, fraction X & 31; weights (32 - fx)(32 - fy), fx (32 - fy), (32 - fx) fy, fx fy; every tap
//   clamped into the frame; result (sum w p + 512) >> 10.
// (OpenCV's table weights are these times 32 with a 15-bit shift: the same integers.)  Each block also adds the
// bytes it wrote to the crop's uint64 sum for the near-black test.
#include "../../include/unetb200.h"

#include <cuda_runtime.h>

#include <cmath>
#include <cstdio>

#include "errors.h"

static_assert(sizeof(unetb200_warp_crop) == 88, "unetb200_warp_crop layout is part of the ABI");

namespace {

constexpr int kWarpTileW = 32, kWarpTileH = 8;   // one thread per output pixel of a 32 x 8 tile
constexpr int kWarpMaxSide = 32767;              // OpenCV keeps source coordinates in int16
constexpr double kWarpMaxCoord = 1 << 19;        // |M00 j|, |M01 i + M02| (and row 2) below 2^19: X fits int32
constexpr unsigned kWarpMaxGridX = 512;

__global__ void __launch_bounds__(kWarpTileW * kWarpTileH) warp_crops_kernel(const unetb200_warp_crop* __restrict__ tab,
                                                                             uint8_t* __restrict__ out,
                                                                             unsigned long long* __restrict__ sums) {
    __shared__ unsigned long long red[kWarpTileW * kWarpTileH / 32];
    const unetb200_warp_crop& c = tab[blockIdx.y];
    const int ow = c.out_w, oh = c.out_h, sw = c.src_w, sh = c.src_h, stride = c.src_stride, pb = c.src_pixel_bytes;
    const double m0 = c.m[0], m1 = c.m[1], m2 = c.m[2], m3 = c.m[3], m4 = c.m[4], m5 = c.m[5];
    const uint8_t* src = reinterpret_cast<const uint8_t*>(c.src);
    uint8_t* dst = out + c.out_off;
    const int tiles_x = (ow + kWarpTileW - 1) / kWarpTileW;
    const int tiles = tiles_x * ((oh + kWarpTileH - 1) / kWarpTileH);
    unsigned long long acc = 0;
    for (int t = blockIdx.x; t < tiles; t += gridDim.x) {      // t advances by a constant: tiles / gridDim.x rounds
        const int ty = t / tiles_x, tx = t - ty * tiles_x;
        const int j = tx * kWarpTileW + static_cast<int>(threadIdx.x % kWarpTileW);
        const int i = ty * kWarpTileH + static_cast<int>(threadIdx.x / kWarpTileW);
        if (j >= ow || i >= oh) continue;
        const double di = static_cast<double>(i), dj = static_cast<double>(j);
        const int X = (__double2int_rn(__dmul_rn(__dadd_rn(__dmul_rn(m1, di), m2), 1024.0)) + 16 +
                       __double2int_rn(__dmul_rn(__dmul_rn(m0, dj), 1024.0))) >> 5;
        const int Y = (__double2int_rn(__dmul_rn(__dadd_rn(__dmul_rn(m4, di), m5), 1024.0)) + 16 +
                       __double2int_rn(__dmul_rn(__dmul_rn(m3, dj), 1024.0))) >> 5;
        const int x0 = X >> 5, fx = X & 31, y0 = Y >> 5, fy = Y & 31;
        const int xa = min(max(x0, 0), sw - 1), xb = min(max(x0 + 1, 0), sw - 1);
        const int ya = min(max(y0, 0), sh - 1), yb = min(max(y0 + 1, 0), sh - 1);
        const int w00 = (32 - fx) * (32 - fy), w01 = fx * (32 - fy), w10 = (32 - fx) * fy, w11 = fx * fy;
        const uint8_t* r0 = src + static_cast<size_t>(ya) * stride * pb;
        const uint8_t* r1 = src + static_cast<size_t>(yb) * stride * pb;
        uint8_t* o = dst + (static_cast<size_t>(i) * ow + j) * 3;
#pragma unroll
        for (int ch = 0; ch < 3; ++ch) {
            const int v = (w00 * __ldg(r0 + xa * pb + ch) + w01 * __ldg(r0 + xb * pb + ch) +
                           w10 * __ldg(r1 + xa * pb + ch) + w11 * __ldg(r1 + xb * pb + ch) + 512) >> 10;
            o[ch] = static_cast<uint8_t>(v);
            acc += static_cast<unsigned>(v);
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned long long tot = 0;
#pragma unroll
        for (int k = 0; k < kWarpTileW * kWarpTileH / 32; ++k) tot += red[k];
        if (tot) atomicAdd(sums + blockIdx.y, tot);
    }
}

// |a i + b| < 2^19 for i in [0, n): a linear function is extreme at an end.  Each of the two rounded terms of X is
// then below 2^29 in magnitude (rounding moves the ends by far less than the factor 2 left to int32), and NaN and
// infinities fail the comparison.
bool coord_ok(double a, double b, int n) {
    const double lo = std::fabs(b), hi = std::fabs(a * (n - 1) + b);
    return lo < kWarpMaxCoord && hi < kWarpMaxCoord;
}

}  // namespace

extern "C" {

int unetb200_warp_crops(const unetb200_warp_crop* table_host, const void* table_dev, int n, uint8_t* out,
                        uint64_t* sums, void* stream) {
    if (!table_host || !table_dev || !out || !sums || n <= 0)
        return ub_fail(UNETB200_EINVAL, "warp_crops: bad argument");
    if (n > 65535) return ub_fail(UNETB200_EINVAL, "warp_crops: at most 65535 crops per call");
    if ((reinterpret_cast<uintptr_t>(table_dev) | reinterpret_cast<uintptr_t>(sums)) & 7)
        return ub_fail(UNETB200_EINVAL, "warp_crops: table and sums must be 8-byte aligned");
    int max_tiles = 0;
    uint64_t end = 0;
    for (int k = 0; k < n; ++k) {
        const unetb200_warp_crop& c = table_host[k];
        char buf[200];
        const char* why = nullptr;
        if (!c.src) why = "null source";
        else if (c.src_h < 1 || c.src_w < 1 || c.src_h > kWarpMaxSide || c.src_w > kWarpMaxSide) why = "source size";
        else if (c.src_stride < c.src_w) why = "source stride below its width";
        else if (c.src_pixel_bytes != 3 && c.src_pixel_bytes != 4) why = "src_pixel_bytes must be 3 or 4";
        else if (c.out_w < 1 || c.out_h < 1 || c.out_w > kWarpMaxSide || c.out_h > kWarpMaxSide) why = "output size";
        else if (c.out_off < end) why = "output overlaps the previous crop (out_off must not decrease)";
        else if (!coord_ok(c.m[0], 0.0, c.out_w) || !coord_ok(c.m[1], c.m[2], c.out_h) ||
                 !coord_ok(c.m[3], 0.0, c.out_w) || !coord_ok(c.m[4], c.m[5], c.out_h))
            why = "matrix maps the crop outside the fixed-point range (|coordinate| < 2^19) or is not finite";
        if (why) {
            snprintf(buf, sizeof buf, "warp_crops: crop %d: %s", k, why);
            return ub_fail(UNETB200_EINVAL, buf);
        }
        end = c.out_off + 3ull * static_cast<uint64_t>(c.out_w) * static_cast<uint64_t>(c.out_h);
        const int tiles = ((c.out_w + kWarpTileW - 1) / kWarpTileW) * ((c.out_h + kWarpTileH - 1) / kWarpTileH);
        max_tiles = tiles > max_tiles ? tiles : max_tiles;
    }
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    cudaError_t e = cudaMemsetAsync(sums, 0, static_cast<size_t>(n) * sizeof(uint64_t), s);
    if (e == cudaSuccess) {
        const dim3 grid(static_cast<unsigned>(max_tiles) < kWarpMaxGridX ? static_cast<unsigned>(max_tiles)
                                                                          : kWarpMaxGridX,
                        static_cast<unsigned>(n));
        warp_crops_kernel<<<grid, kWarpTileW * kWarpTileH, 0, s>>>(
            static_cast<const unetb200_warp_crop*>(table_dev), out, reinterpret_cast<unsigned long long*>(sums));
        e = cudaGetLastError();
    }
    if (e != cudaSuccess) {
        char buf[200];
        snprintf(buf, sizeof buf, "warp_crops: launch failed: %s", cudaGetErrorString(e));
        return ub_fail(UNETB200_ECUDA, buf);
    }
    return UNETB200_OK;
}

}  // extern "C"
