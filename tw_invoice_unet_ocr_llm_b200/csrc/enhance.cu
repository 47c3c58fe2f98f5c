// C ABI of the OCR crop enhancement (include/unetb200.h, "OCR crop enhancement"); kernels in enhance.cuh.
#include "enhance.cuh"

#include <algorithm>
#include <cmath>
#include <cstdio>

#include "errors.h"

static_assert(sizeof(unetb200_enh_crop) == 80, "unetb200_enh_crop layout is part of the ABI");

namespace {

// cv::interpolateCubic (A = -0.75) in float, then saturate_cast<short>(c * INTER_RESIZE_COEF_SCALE)
// (resize.cpp); for fx = 4 the fractional offset only depends on the output coordinate modulo 4.
ub::EnhTaps cubic_taps_x4() {
    ub::EnhTaps t;
    for (int d = 0; d < 4; ++d) {
        float fx = static_cast<float>((d + 0.5) * 0.25 - 0.5);
        const int s = static_cast<int>(std::floor(fx));
        fx -= s;
        const float A = -0.75f;
        float c[4];
        c[0] = ((A * (fx + 1) - 5 * A) * (fx + 1) + 8 * A) * (fx + 1) - 4 * A;
        c[1] = ((A + 2) * fx - (A + 3)) * fx * fx + 1;
        c[2] = ((A + 2) * (1 - fx) - (A + 3)) * (1 - fx) * (1 - fx) + 1;
        c[3] = 1.f - c[0] - c[1] - c[2];
        for (int k = 0; k < 4; ++k) t.t[d][k] = static_cast<int16_t>(std::lrintf(c[k] * 2048.f));
    }
    return t;
}

constexpr int kMaxSide = 8192;          // 4x -> 32768: keeps every int product below 2^31

bool crop_ok(const unetb200_enh_crop& c) {
    return c.h > 0 && c.w > 0 && c.h <= kMaxSide && c.w <= kMaxSide &&
           (c.flags & ~(UNETB200_ENH_SHARPEN | UNETB200_ENH_BLUR | UNETB200_ENH_OTSU)) == 0 && c.clip > 0 &&
           std::isfinite(c.clip) &&
           (c.src_stride == 0 || c.src_stride >= c.w) &&
           (c.src_pixel_bytes == 0 || c.src_pixel_bytes == 3 || c.src_pixel_bytes == 4) &&
           (c.src_stride != 0 || c.src_pixel_bytes != 4);          // packed crops are RGB
}

// what unetb200_enhance_plan derives from h, w and clip alone (enhance_run checks a table against it)
struct EnhGeometry {
    int tile_h, tile_w, clip_count, blocks_x, n_blocks;
};

EnhGeometry enh_geometry(const unetb200_enh_crop& c) {
    const int H = 4 * c.h, W = 4 * c.w;
    // CLAHE_Impl::apply: both dimensions are extended unless both divide the grid
    int eh = H, ew = W;
    if (H % ub::kEnhTiles != 0 || W % ub::kEnhTiles != 0) {
        eh = H + (ub::kEnhTiles - H % ub::kEnhTiles);
        ew = W + (ub::kEnhTiles - W % ub::kEnhTiles);
    }
    EnhGeometry g;
    g.tile_h = eh / ub::kEnhTiles;
    g.tile_w = ew / ub::kEnhTiles;
    const int area = g.tile_h * g.tile_w;
    // CLAHE_Impl::apply: (int)(clipLimit * tileSizeTotal / 256) in double.  No bin of a tile holds more than its
    // area, so a limit at or above the area clips nothing, exactly like any larger one: clamping there keeps the
    // conversion in range (huge or overflowing products) and the LUTs OpenCV's wherever its own int is defined.
    const double limit = std::min(c.clip * area / 256, static_cast<double>(area));
    g.clip_count = std::max(static_cast<int>(limit), 1);
    g.blocks_x = (W + ub::kEnhBlock - 1) / ub::kEnhBlock;
    g.n_blocks = g.blocks_x * ((H + ub::kEnhBlock - 1) / ub::kEnhBlock);
    return g;
}

}  // namespace

extern "C" {

int unetb200_enhance_plan(unetb200_enh_crop* table, int n, uint64_t* src_bytes, uint64_t* out_bytes,
                          uint64_t* workspace_bytes) {
    if (!table || n <= 0 || !src_bytes || !out_bytes || !workspace_bytes)
        return ub_fail(UNETB200_EINVAL, "enhance_plan: bad argument");
    uint64_t so = 0, oo = 0, wo = 0;
    int64_t blocks = 0;
    for (int i = 0; i < n; ++i) {
        unetb200_enh_crop& c = table[i];
        if (!crop_ok(c)) {
            char buf[160];
            snprintf(buf, sizeof buf, "enhance_plan: crop %d invalid (h=%d w=%d flags=%d clip=%g)", i, c.h, c.w,
                     c.flags, c.clip);
            return ub_fail(UNETB200_EINVAL, buf);
        }
        const EnhGeometry g = enh_geometry(c);
        c.tile_h = g.tile_h;
        c.tile_w = g.tile_w;
        c.clip_count = g.clip_count;
        c.blocks_x = g.blocks_x;
        c.n_blocks = g.n_blocks;
        if (blocks + c.n_blocks > 0x7fffffff) return ub_fail(UNETB200_EINVAL, "enhance_plan: batch too large");
        c.first_block = static_cast<int32_t>(blocks);
        blocks += c.n_blocks;
        if (c.src_pixel_bytes == 0) c.src_pixel_bytes = 3;
        if (c.src_stride == 0) {             // packed crop: placed here
            c.src_stride = c.w;
            c.src_off = so;
            so += (static_cast<uint64_t>(3) * c.h * c.w + 15) & ~static_cast<uint64_t>(15);
        }
        c.out_off = oo;
        c.ws_off = wo;
        oo += ub::enh_img_bytes(c.h, c.w);
        wo += ub::enh_ws_bytes(c.h, c.w);
    }
    *src_bytes = so;
    *out_bytes = oo;
    *workspace_bytes = wo;
    return UNETB200_OK;
}

int unetb200_enhance_run(const unetb200_enh_crop* table_host, const void* table_dev, int n,
                         const uint8_t* src_dev, uint8_t* out_dev, void* workspace_dev, void* stream) {
    if (!table_host || !table_dev || n <= 0 || !src_dev || !out_dev || !workspace_dev)  // src_dev: packed crops and/or the frame
        return ub_fail(UNETB200_EINVAL, "enhance_run: bad argument");
    if ((reinterpret_cast<uintptr_t>(out_dev) | reinterpret_cast<uintptr_t>(workspace_dev) |
         reinterpret_cast<uintptr_t>(table_dev)) & 15)
        return ub_fail(UNETB200_EINVAL, "enhance_run: device buffers must be 16-byte aligned");
    // the kernels index shared memory, LUTs and buffers by these fields: every one must be the plan's
    int64_t blocks = 0;
    uint64_t out_bytes = 0, ws_bytes = 0;
    bool any_otsu = false;
    for (int i = 0; i < n; ++i) {
        const unetb200_enh_crop& c = table_host[i];
        const char* bad = nullptr;
        if (!crop_ok(c)) {
            bad = "h, w, flags, clip or source layout invalid";
        } else {
            const EnhGeometry g = enh_geometry(c);
            if (c.src_stride < c.w || c.src_pixel_bytes == 0) bad = "src_stride / src_pixel_bytes not planned";
            else if (c.tile_h != g.tile_h || c.tile_w != g.tile_w) bad = "tile_h / tile_w differ from the plan";
            else if (c.clip_count != g.clip_count) bad = "clip_count differs from the plan";
            else if (c.blocks_x != g.blocks_x || c.n_blocks != g.n_blocks)
                bad = "blocks_x / n_blocks differ from the plan";
            else if (c.first_block != blocks) bad = "first_block differs from the plan";
            else if (c.out_off != out_bytes) bad = "out_off differs from the plan";
            else if (c.ws_off != ws_bytes) bad = "ws_off differs from the plan";
        }
        if (bad) {
            char buf[200];
            snprintf(buf, sizeof buf, "enhance_run: crop %d: %s (table was not produced by unetb200_enhance_plan)",
                     i, bad);
            return ub_fail(UNETB200_EINVAL, buf);
        }
        blocks += c.n_blocks;
        out_bytes += ub::enh_img_bytes(c.h, c.w);
        ws_bytes += ub::enh_ws_bytes(c.h, c.w);
        any_otsu = any_otsu || (c.flags & UNETB200_ENH_OTSU);
    }
    if (blocks > 0x7fffffff || static_cast<int64_t>(n) * ub::kEnhTiles * ub::kEnhTiles > 0x7fffffff)
        return ub_fail(UNETB200_EINVAL, "enhance_run: batch too large");
    static const ub::EnhTaps taps = cubic_taps_x4();
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const auto* tab = static_cast<const unetb200_enh_crop*>(table_dev);
    uint8_t* ws = static_cast<uint8_t*>(workspace_dev);
    const unsigned nb = static_cast<unsigned>(blocks);
    // persistent grid for the upscale: one wave of resident CTAs (SMs x occupancy), each walking a
    // contiguous run of the block list
    int dev = 0, sms = 148, occ = 8;
    if (cudaGetDevice(&dev) == cudaSuccess) {
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, ub::enh_resize_kernel, ub::kEnhResThreads, 0) !=
                cudaSuccess || occ < 1)
            occ = 8;
    }
    const unsigned wave = static_cast<unsigned>(sms) * static_cast<unsigned>(occ);
    const unsigned grid = nb < wave ? nb : wave;
    ub::enh_resize_kernel<<<grid, ub::kEnhResThreads, 0, s>>>(tab, n, static_cast<int>(nb), src_dev, ws, taps);
    ub::enh_lut_kernel<<<static_cast<unsigned>(n) * ub::kEnhTiles * ub::kEnhTiles, ub::kEnhThreads, 0, s>>>(tab, ws);
    ub::enh_clahe_kernel<<<nb, ub::kEnhThreads, 0, s>>>(tab, n, ws, out_dev);
    if (any_otsu) {
        ub::enh_otsu_kernel<<<static_cast<unsigned>(n), ub::kEnhThreads, 0, s>>>(tab, ws);
        const unsigned spans = static_cast<unsigned>((out_bytes + ub::kEnhBinSpan - 1) / ub::kEnhBinSpan);
        ub::enh_binarize_kernel<<<spans, ub::kEnhThreads, 0, s>>>(tab, n, ws, out_dev, out_bytes);
    }
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        char buf[200];
        snprintf(buf, sizeof buf, "enhance_run: launch failed: %s", cudaGetErrorString(e));
        return ub_fail(UNETB200_ECUDA, buf);
    }
    return UNETB200_OK;
}

}  // extern "C"
