// Binary morphology of mask planes (include/unetb200.h, unetb200_mask_morph): erosion and dilation by a kw x kh
// rectangle, opening, closing, and hole filling, bit-exact with cv2.erode / cv2.dilate / cv2.morphologyEx (default
// anchor and border) and scipy.ndimage.binary_fill_holes.  DESIGN.md 6b, "Mask clean-up".
//
// Planes are processed as rows of 32-bit words, pixel x = bit x & 31 of word x >> 5 of its row (wpr = ceil(w / 32)
// words per row): the unetb200_forward_bits layout when w % 32 == 0, which bit-packed input and output use in place.
//
//   mm_pack_kernel    byte planes -> bit rows (non-zero = set)
//   mm_rect_kernel    one erosion / dilation: the horizontal pass of every row of a tile and its vertical halo as it
//                     is staged in shared memory, then the vertical pass over the staged rows
//   mm_unpack_kernel  bit rows -> byte planes of 0 / 1
//
// Opening and closing chain two mm_rect_kernel launches through the workspace.  Hole filling labels the complement
// on the union-find of components.cu (cc_fill_holes).
#include "../../include/unetb200.h"

#include <cuda_runtime.h>

#include <cstdio>

#include "cc_internal.h"
#include "errors.h"

namespace {

constexpr int kMaxK = 63;           // largest element side: each side of the window reaches at most 31 pixels
constexpr int kTileRows = 64;       // output rows of one mm_rect_kernel block
constexpr int kColWords = 32;       // word columns of one mm_rect_kernel block (threadIdx.x)
constexpr int kRowThreads = 8;      // threadIdx.y

struct Rows {
    int h, w;
    int wpr;                        // words per row
    uint32_t tail;                  // valid bits of the last word of a row (all ones when w % 32 == 0)
};

// AND (erosion) or OR (dilation); the border value is the identity of the operation
template <bool DIL>
__device__ __forceinline__ uint32_t op32(uint32_t a, uint32_t b) { return DIL ? (a | b) : (a & b); }
template <bool DIL>
__device__ __forceinline__ unsigned long long op64(unsigned long long a, unsigned long long b) {
    return DIL ? (a | b) : (a & b);
}

// Word k of a row with the border rule applied: words outside the row and the pad bits past w are the identity.
template <bool DIL>
__device__ __forceinline__ uint32_t row_word(const uint32_t* __restrict__ row, int k, const Rows& g) {
    const uint32_t fill = DIL ? 0u : 0xffffffffu;
    if (k < 0 || k >= g.wpr) return fill;
    const uint32_t v = __ldg(row + k);
    if (k != g.wpr - 1) return v;
    return DIL ? (v & g.tail) : (v | ~g.tail);
}

// Horizontal pass of word k: bit j = op of pixels 32k + j - ax .. 32k + j + r (ax = kw / 2, r = kw - 1 - ax, both
// <= 31).  Right reach: the 64-bit pair (right word : word) shifted down by 1, 2, 4, ... combines spans that double
// each step (s has span `sp` at every bit), then one last shift by r + 1 - sp closes the window; only bits 0..31
// are kept, and they read bits up to 31 + r <= 62, so the zeros shifted in from the top never reach them.  The left
// reach is the mirror image on (word : left word), shifting up and keeping bits 32..63.
template <bool DIL>
__device__ __forceinline__ uint32_t hpass(const uint32_t* __restrict__ row, int k, const Rows& g, int kw) {
    const unsigned long long L = row_word<DIL>(row, k - 1, g), C = row_word<DIL>(row, k, g),
                             R = row_word<DIL>(row, k + 1, g);
    const int ax = kw >> 1, r = kw - 1 - ax;
    unsigned long long s = (R << 32) | C;
    int sp = 1;
    while (2 * sp <= r + 1) {                          // sp doubles: at most 5 rounds
        s = op64<DIL>(s, s >> sp);
        sp <<= 1;
    }
    s = op64<DIL>(s, s >> (r + 1 - sp));
    unsigned long long u = (C << 32) | L;
    sp = 1;
    while (2 * sp <= ax + 1) {
        u = op64<DIL>(u, u << sp);
        sp <<= 1;
    }
    u = op64<DIL>(u, u << (ax + 1 - sp));
    return op32<DIL>(static_cast<uint32_t>(s), static_cast<uint32_t>(u >> 32));
}

__global__ void __launch_bounds__(256) mm_pack_kernel(const uint8_t* __restrict__ mask, long long n_words, Rows g,
                                                      uint32_t* __restrict__ bits) {
    const long long t = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    const long long word = t >> 5;                       // one warp per word, one lane per pixel
    if (word >= n_words) return;                         // whole warps leave together
    const long long row = word / g.wpr;                  // plane * h + y
    const int x = static_cast<int>(word - row * g.wpr) * 32 + static_cast<int>(threadIdx.x & 31);
    const bool on = x < g.w && mask[row * g.w + x] != 0;
    const uint32_t v = __ballot_sync(0xffffffffu, on);
    if ((threadIdx.x & 31) == 0) bits[word] = v;
}

__global__ void __launch_bounds__(256) mm_unpack_kernel(const uint32_t* __restrict__ bits, long long n_px, Rows g,
                                                        uint8_t* __restrict__ out) {
    const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= n_px) return;
    const long long row = i / g.w;
    const int x = static_cast<int>(i - row * g.w);
    out[i] = static_cast<uint8_t>((__ldg(bits + row * g.wpr + (x >> 5)) >> (x & 31)) & 1u);
}

// One block = kColWords word columns x kTileRows output rows of one plane.  Staging: rows y0 - ay ..
// y0 + kTileRows - 1 + (kh - 1 - ay) after the horizontal pass (rows outside the plane: the identity) in buf[0].
// Vertical pass by doubling: after the round of span sp, row i holds op of staged rows i .. i + 2 sp - 1; with
// sp = the largest power of two <= kh, output row t = op(row t, row t + kh - sp), two windows of sp rows that
// overlap (kh - sp < sp) and together cover staged rows t .. t + kh - 1.  Every thread runs every round (the loop
// bounds depend on threadIdx.y only), so the barriers are uniform.
template <bool DIL>
__global__ void __launch_bounds__(kColWords * kRowThreads) mm_rect_kernel(const uint32_t* __restrict__ src,
                                                                          uint32_t* __restrict__ dst, Rows g,
                                                                          int kw, int kh, int col_blocks,
                                                                          int row_blocks) {
    __shared__ uint32_t buf[2][kTileRows + kMaxK - 1][kColWords];
    const int cb = blockIdx.x % col_blocks;
    const int rest = blockIdx.x / col_blocks;
    const int rb = rest % row_blocks, p = rest / row_blocks;
    const int lane = threadIdx.x, ty = threadIdx.y;
    const int k = cb * kColWords + lane;
    const bool active = k < g.wpr;
    const int y0 = rb * kTileRows, ay = kh >> 1;
    const size_t plane = static_cast<size_t>(p) * g.h * g.wpr;
    const int staged = kTileRows + kh - 1;
    for (int i = ty; i < staged; i += kRowThreads) {
        const int y = y0 - ay + i;
        uint32_t v = DIL ? 0u : 0xffffffffu;
        if (active && y >= 0 && y < g.h) v = hpass<DIL>(src + plane + static_cast<size_t>(y) * g.wpr, k, g, kw);
        buf[0][i][lane] = v;
    }
    __syncthreads();
    int cur = 0, len = staged, sp = 1;
    while (2 * sp <= kh) {                               // sp doubles: at most 5 rounds
        for (int i = ty; i < len - sp; i += kRowThreads)
            buf[cur ^ 1][i][lane] = op32<DIL>(buf[cur][i][lane], buf[cur][i + sp][lane]);
        len -= sp;
        sp <<= 1;
        cur ^= 1;
        __syncthreads();
    }
    for (int t = ty; t < kTileRows; t += kRowThreads) {
        const int y = y0 + t;
        if (active && y < g.h)
            dst[plane + static_cast<size_t>(y) * g.wpr + k] = op32<DIL>(buf[cur][t][lane], buf[cur][t + kh - sp][lane]);
    }
}

bool rows_of(int h, int w, Rows* g) {
    if (h <= 0 || w <= 0 || static_cast<long long>(h) * w >= (1LL << 31)) return false;
    g->h = h;
    g->w = w;
    g->wpr = (w + 31) / 32;
    g->tail = (w & 31) ? (1u << (w & 31)) - 1u : 0xffffffffu;
    return true;
}

// Bytes of one bit-row region of the workspace (16-byte multiple)
unsigned long long region_bytes(int n_planes, const Rows& g) {
    return (static_cast<unsigned long long>(n_planes) * g.h * g.wpr * 4ull + 15ull) & ~15ull;
}

bool overlap(const void* a, unsigned long long na, const void* b, unsigned long long nb) {
    const uintptr_t x = reinterpret_cast<uintptr_t>(a), y = reinterpret_cast<uintptr_t>(b);
    return x < y + nb && y < x + na;
}

}  // namespace

extern "C" {

uint64_t unetb200_morph_workspace_bytes(int n_planes, int h, int w, int op) {
    Rows g;
    if (n_planes <= 0 || !rows_of(h, w, &g)) return 0;
    if (op == UNETB200_MORPH_FILL_HOLES) return unetb200_components_workspace_bytes(n_planes, h, w);
    if (op < UNETB200_MORPH_ERODE || op > UNETB200_MORPH_CLOSE) return 0;
    return 2 * region_bytes(n_planes, g);
}

int unetb200_mask_morph(const uint8_t* in, int in_packed, uint8_t* out, int out_packed, int n_planes, int h, int w,
                        int op, int kw, int kh, void* workspace, uint64_t workspace_bytes, void* stream) {
    char buf[240];
    auto fail = [&](int code, const char* msg) {
        snprintf(buf, sizeof buf, "mask_morph: %s", msg);
        return ub_fail(code, buf);
    };
    Rows g;
    if (!in || !out || !workspace)
        return fail(UNETB200_EINVAL, "null pointer");
    if (op < UNETB200_MORPH_ERODE || op > UNETB200_MORPH_FILL_HOLES)
        return fail(UNETB200_EINVAL, "op must be one of UNETB200_MORPH_ERODE .. UNETB200_MORPH_FILL_HOLES");
    if (op != UNETB200_MORPH_FILL_HOLES && (kw < 1 || kw > kMaxK || kh < 1 || kh > kMaxK))
        return fail(UNETB200_EINVAL, "kw and kh must be in [1, 63]");
    if ((in_packed != 0 && in_packed != 1) || (out_packed != 0 && out_packed != 1))
        return fail(UNETB200_EINVAL, "in_packed and out_packed must be 0 or 1");
    if (n_planes <= 0 || !rows_of(h, w, &g))
        return fail(UNETB200_EINVAL, "bad size (n_planes, h, w >= 1 and h * w < 2^31)");
    if ((in_packed || out_packed) && (w & 31))
        return fail(UNETB200_EINVAL, "bit-packed planes need w % 32 == 0");
    if (((in_packed ? reinterpret_cast<uintptr_t>(in) : 0) | (out_packed ? reinterpret_cast<uintptr_t>(out) : 0)) & 3 ||
        (reinterpret_cast<uintptr_t>(workspace) & 15))
        return fail(UNETB200_EINVAL, "misaligned pointer (bit-packed planes 4-byte aligned, workspace 16-byte aligned)");
    const uint64_t need = unetb200_morph_workspace_bytes(n_planes, h, w, op);
    if (need == 0)
        return fail(UNETB200_EINVAL, "bad size (n_planes, h, w >= 1 and h * w < 2^31)");
    if (workspace_bytes < need)
        return fail(UNETB200_ENOMEM, "workspace smaller than unetb200_morph_workspace_bytes");
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    if (op == UNETB200_MORPH_FILL_HOLES)
        return cc_fill_holes("mask_morph", in, in_packed, out, out_packed, n_planes, h, w, workspace, s);

    const long long n_words = static_cast<long long>(n_planes) * h * g.wpr;
    const long long n_px = static_cast<long long>(n_planes) * h * w;
    const int col_blocks = (g.wpr + kColWords - 1) / kColWords, row_blocks = (h + kTileRows - 1) / kTileRows;
    const long long rect_blocks = static_cast<long long>(col_blocks) * row_blocks * n_planes;
    if (rect_blocks >= (1LL << 31) || (n_words * 32 + 255) / 256 >= (1LL << 31) || (n_px + 255) / 256 >= (1LL << 31))
        return fail(UNETB200_EINVAL, "batch too large");

    uint32_t* a = static_cast<uint32_t*>(workspace);
    uint32_t* b = reinterpret_cast<uint32_t*>(static_cast<char*>(workspace) + region_bytes(n_planes, g));
    // The first pass reads the input and every later one reads the workspace, so in-place calls work: bit-packed
    // input that overlaps the output is copied to the workspace first, byte input is packed there anyway.
    const uint32_t* cur = reinterpret_cast<const uint32_t*>(in);
    const unsigned long long in_bytes = in_packed ? n_words * 4ull : static_cast<unsigned long long>(n_px);
    const unsigned long long out_bytes = out_packed ? n_words * 4ull : static_cast<unsigned long long>(n_px);
    if (!in_packed) {
        mm_pack_kernel<<<static_cast<unsigned>((n_words * 32 + 255) / 256), 256, 0, s>>>(in, n_words, g, a);
        cur = a;
    } else if (overlap(in, in_bytes, out, out_bytes)) {
        const cudaError_t e = cudaMemcpyAsync(a, in, n_words * 4ull, cudaMemcpyDeviceToDevice, s);
        if (e != cudaSuccess) {
            snprintf(buf, sizeof buf, "mask_morph: copy failed: %s", cudaGetErrorString(e));
            return ub_fail(UNETB200_ECUDA, buf);
        }
        cur = a;
    }
    // erode / dilate: one pass; open = erode then dilate; close = dilate then erode
    const bool dil[2] = {op == UNETB200_MORPH_DILATE || op == UNETB200_MORPH_CLOSE, op == UNETB200_MORPH_OPEN};
    const int passes = (op == UNETB200_MORPH_OPEN || op == UNETB200_MORPH_CLOSE) ? 2 : 1;
    const dim3 block(kColWords, kRowThreads);
    for (int j = 0; j < passes; ++j) {
        uint32_t* dst = (j == passes - 1 && out_packed) ? reinterpret_cast<uint32_t*>(out) : (cur == a ? b : a);
        if (dil[j])
            mm_rect_kernel<true><<<static_cast<unsigned>(rect_blocks), block, 0, s>>>(cur, dst, g, kw, kh, col_blocks,
                                                                                    row_blocks);
        else
            mm_rect_kernel<false><<<static_cast<unsigned>(rect_blocks), block, 0, s>>>(cur, dst, g, kw, kh, col_blocks,
                                                                                     row_blocks);
        cur = dst;
    }
    if (!out_packed)
        mm_unpack_kernel<<<static_cast<unsigned>((n_px + 255) / 256), 256, 0, s>>>(cur, n_px, g, out);
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        snprintf(buf, sizeof buf, "mask_morph: launch failed: %s", cudaGetErrorString(e));
        return ub_fail(UNETB200_ECUDA, buf);
    }
    return UNETB200_OK;
}

}  // extern "C"
