// Connected-component labelling of binary planes (include/unetb200.h, unetb200_mask_components): block-based
// union-find (Playne & Hawick 2018; Allegretti et al. 2019, BUF).  Per call, in stream order:
//
//   cc_pack_kernel     byte masks -> one bit per pixel, plane-contiguous (bit i & 31 of word i >> 5 is pixel
//                      i = y * w + x); bit-packed input with w % 32 == 0 already has this layout and is read as is
//   cc_local_kernel    union-find inside a 32 x 16 tile in shared memory; writes parent[i] = the tile-local root
//   cc_merge_kernel    unions across tile borders with atomicMin on the global parents
//   cc_flatten_kernel  parent[i] = root of i; counts the roots of every 1024-pixel raster segment
//   cc_scan_kernel     exclusive scan of the segment counts of a plane; n_comps[plane] = total
//   cc_number_kernel   numbers the roots in raster order (root entry := -(id + 2)), initialises their statistics
//   cc_stats_kernel    labels (optional) + extents and counts by integer atomics, aggregated per warp and id
//   cc_select_kernel   the K largest components of each plane (count descending, label ascending)
//
// Every link points to a smaller raster index (parent[i] <= i), so the root of a component is its first pixel in
// raster order and numbering the roots in raster order gives scipy.ndimage.label's labels.  All statistics are
// integer min / max / add, so every output is independent of scheduling.
#include "../../include/unetb200.h"

#include <cuda_runtime.h>

#include <cstdio>

#include "errors.h"

namespace {

constexpr int kTileW = 32, kTileH = 16;        // cc_local_kernel: one thread per pixel of a tile
constexpr int kSeg = 1024;                     // raster pixels per root-count segment
constexpr int kSegThreads = 256;
constexpr int kMaxK = 16;
constexpr int kBg = -1;                        // parent entry of a background pixel

struct Plane {
    int h, w, n;          // n = h * w
    int wpp;              // bit words per plane
    int cap;              // statistics rows per plane: ceil(n / 2) bounds the components of a plane
    int nseg;             // root-count segments per plane
};

// Workspace (int32 units, every region back to back): parent [P][n], statistics 5 x [P][cap] (xmin, xmax, ymin,
// ymax, count), segment counts [P][nseg], bits [P][wpp] (byte input only).
struct Work {
    int* parent;
    int *xmin, *xmax, *ymin, *ymax, *count;
    int* seg;
    uint32_t* bits;
};

__device__ __forceinline__ bool bit_at(const uint32_t* __restrict__ bits, int i) {
    return (__ldg(bits + (i >> 5)) >> (i & 31)) & 1u;
}

// Root of `a`.  Invariant: s[x] <= x for every foreground x, so the index strictly decreases until it reaches a
// root (s[x] == x); the loop ends after at most `a` steps whatever other threads write meanwhile.
__device__ __forceinline__ int find_root(const volatile int* s, int a) {
    int p = s[a];
    while (p < a) {
        a = p;
        p = s[a];
    }
    return a;
}

// Joins the trees of a and b (both foreground).  Every write is atomicMin(&s[b], a) with a < b, which keeps
// s[x] <= x.  Each round either ends or replaces the larger of (a, b) by a strictly smaller index (old < b), and
// find_root never increases an index, so max(a, b) strictly decreases: at most max(a, b) rounds, independent of
// other threads.  When the atomicMin finds b already linked (old != b), b's previous parent `old` is joined with a
// in the next round, so no link is lost.
__device__ __forceinline__ void unite(int* s, int a, int b) {
    for (;;) {
        a = find_root(s, a);
        b = find_root(s, b);
        if (a == b) return;
        if (a > b) { const int t = a; a = b; b = t; }
        const int old = atomicMin(s + b, a);
        if (old == b) return;
        b = old;
    }
}

__global__ void __launch_bounds__(256) cc_pack_kernel(const uint8_t* __restrict__ mask, int n_planes, Plane g,
                                                      uint32_t* __restrict__ bits) {
    const long long t = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    const long long word = t >> 5;                       // one warp per word, one lane per pixel
    if (word >= static_cast<long long>(n_planes) * g.wpp) return;     // whole warps leave together
    const int p = static_cast<int>(word / g.wpp), wi = static_cast<int>(word - static_cast<long long>(p) * g.wpp);
    const int i = (wi << 5) + static_cast<int>(threadIdx.x & 31);
    const bool on = i < g.n && mask[static_cast<size_t>(p) * g.n + i] != 0;
    const uint32_t v = __ballot_sync(0xffffffffu, on);
    if ((threadIdx.x & 31) == 0) bits[word] = v;
}

template <int CONN>
__global__ void __launch_bounds__(kTileW * kTileH) cc_local_kernel(const uint32_t* __restrict__ bits, Plane g,
                                                                   int tiles_x, int tiles_per_plane,
                                                                   int* __restrict__ parent) {
    __shared__ int s[kTileW * kTileH];
    const int p = blockIdx.x / tiles_per_plane, tile = blockIdx.x - p * tiles_per_plane;
    const int ty = tile / tiles_x, tx = tile - ty * tiles_x;
    const int lx = threadIdx.x % kTileW, ly = threadIdx.x / kTileW, l = threadIdx.x;
    const int x = tx * kTileW + lx, y = ty * kTileH + ly;
    const uint32_t* pb = bits + static_cast<size_t>(p) * g.wpp;
    const bool fg = x < g.w && y < g.h && bit_at(pb, y * g.w + x);
    // local index l = ly * 32 + lx orders the tile's pixels as their raster indices do
    s[l] = fg ? l : kBg;
    __syncthreads();
    if (fg) {
        const bool left = lx > 0 && s[l - 1] != kBg;
        const bool up = ly > 0 && s[l - kTileW] != kBg;
        if (left) unite(s, l - 1, l);
        if (up) unite(s, l - kTileW, l);
        if (CONN == 8 && !up && ly > 0) {            // a set up neighbour already joins up-left and up-right
            if (lx > 0 && s[l - kTileW - 1] != kBg) unite(s, l - kTileW - 1, l);
            if (lx < kTileW - 1 && s[l - kTileW + 1] != kBg) unite(s, l - kTileW + 1, l);
        }
    }
    __syncthreads();
    if (x < g.w && y < g.h) {
        int v = kBg;
        if (fg) {
            const int r = find_root(s, l);
            v = (ty * kTileH + r / kTileW) * g.w + tx * kTileW + r % kTileW;
        }
        parent[static_cast<size_t>(p) * g.n + y * g.w + x] = v;
    }
}

// One thread per pixel of a tile's top row (32), left column (rows 1..15) and right column (rows 1..15): each
// joins its backward neighbours (left, up, and for 8-connectivity up-left, up-right) that lie in another tile.
// Every adjacent pair of pixels is a backward pair of exactly one of them, and every backward neighbour in
// another tile belongs to one of these border pixels.
template <int CONN>
__global__ void __launch_bounds__(256) cc_merge_kernel(const uint32_t* __restrict__ bits, Plane g, int tiles_x,
                                                       int tiles_per_plane, long long n_threads,
                                                       int* __restrict__ parent) {
    const long long t = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (t >= n_threads) return;
    const int k = static_cast<int>(t & 63);
    const long long tl = t >> 6;
    const int p = static_cast<int>(tl / tiles_per_plane), tile = static_cast<int>(tl - static_cast<long long>(p) * tiles_per_plane);
    const int ty = tile / tiles_x, tx = tile - ty * tiles_x;
    int x, y;
    if (k < kTileW) { x = tx * kTileW + k; y = ty * kTileH; }
    else if (k < kTileW + kTileH) { x = tx * kTileW; y = ty * kTileH + k - kTileW; if (k == kTileW) return; }
    else { x = tx * kTileW + kTileW - 1; y = ty * kTileH + k - kTileW - kTileH; if (k == kTileW + kTileH || CONN == 4) return; }
    if (x >= g.w || y >= g.h) return;
    const uint32_t* pb = bits + static_cast<size_t>(p) * g.wpp;
    const int i = y * g.w + x;
    if (!bit_at(pb, i)) return;
    int* par = parent + static_cast<size_t>(p) * g.n;
    const int dx[4] = {-1, 0, -1, 1}, dy[4] = {0, -1, -1, -1};
#pragma unroll
    for (int d = 0; d < (CONN == 8 ? 4 : 2); ++d) {
        const int nx = x + dx[d], ny = y + dy[d];
        if (nx < 0 || ny < 0 || nx >= g.w) continue;
        if ((nx / kTileW) == tx && (ny / kTileH) == ty) continue;     // same tile: joined by cc_local_kernel
        const int j = ny * g.w + nx;
        if (bit_at(pb, j)) unite(par, j, i);
    }
}

__device__ __forceinline__ int block_sum_256(int v, int* red) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
    __syncthreads();
    int tot = 0;
#pragma unroll
    for (int wi = 0; wi < kSegThreads / 32; ++wi) tot += red[wi];
    __syncthreads();
    return tot;
}

// One block per segment: parent[i] := root of i (only the own entry is written; every value written is an
// ancestor of i, so concurrent find_root walks stay valid), then the segment's root count.
__global__ void __launch_bounds__(kSegThreads) cc_flatten_kernel(Plane g, int* __restrict__ parent,
                                                                 int* __restrict__ seg) {
    __shared__ int red[kSegThreads / 32];
    const int p = blockIdx.x / g.nseg, sg = blockIdx.x - p * g.nseg;
    int* par = parent + static_cast<size_t>(p) * g.n;
    int roots = 0;
    for (int k = threadIdx.x; k < kSeg; k += kSegThreads) {
        const int i = sg * kSeg + k;
        if (i >= g.n) break;
        const int v = par[i];
        if (v == kBg) continue;
        const int r = find_root(par, i);
        if (r != v) par[i] = r;
        roots += r == i;
    }
    const int tot = block_sum_256(roots, red);
    if (threadIdx.x == 0) seg[static_cast<size_t>(p) * g.nseg + sg] = tot;
}

// One block per plane: exclusive scan of the segment counts in place; n_comps[plane] = the total.
__global__ void __launch_bounds__(1024) cc_scan_kernel(Plane g, int* __restrict__ seg, int32_t* __restrict__ n_comps) {
    __shared__ int warp_tot[32];
    int* sp = seg + static_cast<size_t>(blockIdx.x) * g.nseg;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    int base = 0;
    for (int c0 = 0; c0 < g.nseg; c0 += 1024) {        // c0 advances by a constant: nseg / 1024 + 1 rounds
        const int c = c0 + threadIdx.x;
        const int v = c < g.nseg ? sp[c] : 0;
        int incl = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int u = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += u;
        }
        if (lane == 31) warp_tot[wid] = incl;
        __syncthreads();
        int before = 0, all = 0;
        for (int wi = 0; wi < 32; ++wi) {
            if (wi < wid) before += warp_tot[wi];
            all += warp_tot[wi];
        }
        if (c < g.nseg) sp[c] = base + before + incl - v;
        base += all;
        __syncthreads();
    }
    if (threadIdx.x == 0) n_comps[blockIdx.x] = base;
}

// One block per segment: the roots of the segment in raster order get ids seg_offset, seg_offset + 1, ...; a
// root's parent entry becomes -(id + 2) (background stays -1) and its statistics start at its own pixel.
__global__ void __launch_bounds__(kSegThreads) cc_number_kernel(Plane g, int* __restrict__ parent,
                                                                const int* __restrict__ seg, Work wk) {
    __shared__ int warp_cnt[kSegThreads / 32];
    const int p = blockIdx.x / g.nseg, sg = blockIdx.x - p * g.nseg;
    int* par = parent + static_cast<size_t>(p) * g.n;
    int base = seg[static_cast<size_t>(p) * g.nseg + sg];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    for (int k0 = 0; k0 < kSeg; k0 += kSegThreads) {
        const int i = sg * kSeg + k0 + threadIdx.x;
        const bool root = i < g.n && par[i] == i;
        const uint32_t b = __ballot_sync(0xffffffffu, root);
        if (lane == 0) warp_cnt[wid] = __popc(b);
        __syncthreads();
        int before = 0, all = 0;
#pragma unroll
        for (int wi = 0; wi < kSegThreads / 32; ++wi) {
            if (wi < wid) before += warp_cnt[wi];
            all += warp_cnt[wi];
        }
        if (root) {
            const int id = base + before + __popc(b & ((1u << lane) - 1u));
            if (id < g.cap) {                        // always: a plane has at most ceil(n / 2) components
                par[i] = -(id + 2);
                const size_t o = static_cast<size_t>(p) * g.cap + id;
                const int y = i / g.w, x = i - y * g.w;
                wk.xmin[o] = x; wk.xmax[o] = x; wk.ymin[o] = y; wk.ymax[o] = y; wk.count[o] = 0;
            }
        }
        base += all;
        __syncthreads();
    }
}

// One warp per row, 32 columns per step.  Lanes holding the same id (__match_any_sync) add their pixels with one
// set of atomics from the lowest such lane: the group lies in one row, so its extents are its first and last lane.
__global__ void __launch_bounds__(256) cc_stats_kernel(Plane g, int n_rows, const int* __restrict__ parent,
                                                       Work wk, int32_t* __restrict__ labels) {
    const long long row = static_cast<long long>(blockIdx.x) * 8 + (threadIdx.x >> 5);
    if (row >= n_rows) return;                                       // whole warps leave together
    const int p = static_cast<int>(row / g.h), y = static_cast<int>(row - static_cast<long long>(p) * g.h);
    const int lane = threadIdx.x & 31;
    const int* par = parent + static_cast<size_t>(p) * g.n;
    const size_t so = static_cast<size_t>(p) * g.cap;
    for (int x0 = 0; x0 < g.w; x0 += 32) {
        const int x = x0 + lane;
        int id = -1;
        if (x < g.w) {
            const int v = par[y * g.w + x];
            if (v != kBg) id = v < kBg ? -v - 2 : -par[v] - 2;
            if (labels) labels[static_cast<size_t>(p) * g.n + y * g.w + x] = id + 1;
        }
        const uint32_t grp = __match_any_sync(0xffffffffu, id);
        if (id >= 0 && lane == __ffs(grp) - 1) {
            const size_t o = so + id;
            atomicMin(wk.xmin + o, x);
            atomicMax(wk.xmax + o, x0 + 31 - __clz(grp));
            atomicMax(wk.ymax + o, y);
            atomicAdd(wk.count + o, __popc(grp));
        }
    }
}

// 64-bit sort key: count descending, then label ascending
__device__ __forceinline__ unsigned long long comp_key(int count, int id) {
    return (static_cast<unsigned long long>(count) << 32) | (0xffffffffu - static_cast<uint32_t>(id));
}

// One block per plane: every thread keeps the 16 largest keys of its share in registers (descending, fully
// unrolled insertion), then a tree of pairwise merges in shared memory leaves the plane's 16 largest in list 0.
// Keys are unique per plane (the id is part of the key), so the result does not depend on the order of work.
__global__ void __launch_bounds__(256) cc_select_kernel(Plane g, Work wk, const int32_t* __restrict__ n_comps, int k_out,
                                                        int32_t* __restrict__ comps) {
    __shared__ unsigned long long lists[256][kMaxK];
    const int p = blockIdx.x;
    const int n = min(n_comps[p], g.cap);
    const size_t so = static_cast<size_t>(p) * g.cap;
    unsigned long long top[kMaxK];
#pragma unroll
    for (int j = 0; j < kMaxK; ++j) top[j] = 0;      // count >= 1 for every component: 0 never wins
    for (int id = threadIdx.x; id < n; id += 256) {
        unsigned long long key = comp_key(wk.count[so + id], id);
        if (key <= top[kMaxK - 1]) continue;
#pragma unroll
        for (int j = 0; j < kMaxK; ++j) {            // insert: the larger of (top[j], key) stays, the other moves down
            const unsigned long long hi = top[j] > key ? top[j] : key, lo = top[j] > key ? key : top[j];
            top[j] = hi;
            key = lo;
        }
    }
#pragma unroll
    for (int j = 0; j < kMaxK; ++j) lists[threadIdx.x][j] = top[j];
    __syncthreads();
    for (int half = 128; half > 0; half >>= 1) {     // half halves each round: 8 rounds
        if (static_cast<int>(threadIdx.x) < half) {
            const unsigned long long* a = lists[threadIdx.x];
            const unsigned long long* b = lists[threadIdx.x + half];
            int ia = 0, ib = 0;
#pragma unroll
            for (int j = 0; j < kMaxK; ++j) top[j] = a[ia] >= b[ib] ? a[ia++] : b[ib++];   // ia + ib == j < 16
        }
        __syncthreads();
        if (static_cast<int>(threadIdx.x) < half) {
#pragma unroll
            for (int j = 0; j < kMaxK; ++j) lists[threadIdx.x][j] = top[j];
        }
        __syncthreads();
    }
    if (static_cast<int>(threadIdx.x) < k_out) {
        int32_t* o = comps + (static_cast<size_t>(p) * k_out + threadIdx.x) * 6;
        const unsigned long long key = lists[0][threadIdx.x];
        if (key == 0) {
            o[0] = g.w; o[1] = -1; o[2] = g.h; o[3] = -1; o[4] = 0; o[5] = 0;
        } else {
            const int id = static_cast<int>(0xffffffffu - static_cast<uint32_t>(key));
            const size_t s = so + id;
            o[0] = wk.xmin[s]; o[1] = wk.xmax[s]; o[2] = wk.ymin[s]; o[3] = wk.ymax[s]; o[4] = wk.count[s];
            o[5] = id + 1;
        }
    }
}

bool plane_of(int h, int w, Plane* g) {
    if (h <= 0 || w <= 0 || static_cast<long long>(h) * w >= (1LL << 31)) return false;
    g->h = h;
    g->w = w;
    g->n = h * w;
    g->wpp = static_cast<int>((static_cast<long long>(g->n) + 31) / 32);
    g->cap = static_cast<int>((static_cast<long long>(g->n) + 1) / 2);
    g->nseg = static_cast<int>((static_cast<long long>(g->n) + kSeg - 1) / kSeg);
    return true;
}

// int32 words of the workspace of n_planes planes
unsigned long long work_words(int n_planes, const Plane& g) {
    return static_cast<unsigned long long>(n_planes) *
           (static_cast<unsigned long long>(g.n) + 5ull * g.cap + g.nseg + g.wpp);
}

}  // namespace

extern "C" {

uint64_t unetb200_components_workspace_bytes(int n_planes, int h, int w) {
    Plane g;
    if (n_planes <= 0 || !plane_of(h, w, &g)) return 0;
    return 4ull * work_words(n_planes, g);
}

int unetb200_mask_components(const uint8_t* mask, int packed, int n_planes, int h, int w, int connectivity,
                             int max_components, int32_t* labels, int32_t* comps, int32_t* n_comps, void* workspace,
                             uint64_t workspace_bytes, void* stream) {
    Plane g;
    if (!mask || !comps || !n_comps || !workspace)
        return ub_fail(UNETB200_EINVAL, "mask_components: null pointer");
    if (connectivity != 4 && connectivity != 8)
        return ub_fail(UNETB200_EINVAL, "mask_components: connectivity must be 4 or 8");
    if (max_components < 1 || max_components > kMaxK)
        return ub_fail(UNETB200_EINVAL, "mask_components: max_components must be in [1, 16]");
    if (packed != 0 && packed != 1)
        return ub_fail(UNETB200_EINVAL, "mask_components: packed must be 0 or 1");
    if (n_planes <= 0 || !plane_of(h, w, &g))
        return ub_fail(UNETB200_EINVAL, "mask_components: bad size (n_planes, h, w >= 1 and h * w < 2^31)");
    if (packed && (w & 31))
        return ub_fail(UNETB200_EINVAL, "mask_components: bit-packed planes need w % 32 == 0");
    if (((packed ? reinterpret_cast<uintptr_t>(mask) : 0) | reinterpret_cast<uintptr_t>(labels) |
         reinterpret_cast<uintptr_t>(comps) | reinterpret_cast<uintptr_t>(n_comps)) & 3 ||
        (reinterpret_cast<uintptr_t>(workspace) & 15))
        return ub_fail(UNETB200_EINVAL, "mask_components: misaligned pointer (int32 outputs and bit-packed planes "
                                        "4-byte aligned, workspace 16-byte aligned)");
    if (workspace_bytes < 4ull * work_words(n_planes, g))
        return ub_fail(UNETB200_ENOMEM, "mask_components: workspace smaller than unetb200_components_workspace_bytes");
    const int tiles_x = (w + kTileW - 1) / kTileW, tiles_y = (h + kTileH - 1) / kTileH;
    const long long tiles = static_cast<long long>(tiles_x) * tiles_y;
    const long long n_rows = static_cast<long long>(n_planes) * h;
    const long long seg_blocks = static_cast<long long>(n_planes) * g.nseg;
    const long long pack_blocks = (static_cast<long long>(n_planes) * g.wpp * 32 + 255) / 256;
    if (tiles * n_planes >= (1LL << 31) || n_rows >= (1LL << 31) || seg_blocks >= (1LL << 31) ||
        pack_blocks >= (1LL << 31))
        return ub_fail(UNETB200_EINVAL, "mask_components: batch too large");

    int* base = static_cast<int*>(workspace);
    const size_t pn = static_cast<size_t>(n_planes) * g.n, pc = static_cast<size_t>(n_planes) * g.cap;
    Work wk;
    wk.parent = base;
    wk.xmin = wk.parent + pn;
    wk.xmax = wk.xmin + pc;
    wk.ymin = wk.xmax + pc;
    wk.ymax = wk.ymin + pc;
    wk.count = wk.ymax + pc;
    wk.seg = wk.count + pc;
    wk.bits = reinterpret_cast<uint32_t*>(wk.seg + static_cast<size_t>(n_planes) * g.nseg);

    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const uint32_t* bits = wk.bits;
    if (packed) {
        bits = reinterpret_cast<const uint32_t*>(mask);  // [h][w/8] with w % 32 == 0 is the plane-contiguous layout
    } else {
        cc_pack_kernel<<<static_cast<unsigned>(pack_blocks), 256, 0, s>>>(mask, n_planes, g, wk.bits);
    }
    const int tpp = static_cast<int>(tiles);
    const unsigned local_blocks = static_cast<unsigned>(tiles * n_planes);
    const long long merge_threads = tiles * n_planes * 64;
    const unsigned merge_blocks = static_cast<unsigned>((merge_threads + 255) / 256);
    if (connectivity == 4) {
        cc_local_kernel<4><<<local_blocks, kTileW * kTileH, 0, s>>>(bits, g, tiles_x, tpp, wk.parent);
        cc_merge_kernel<4><<<merge_blocks, 256, 0, s>>>(bits, g, tiles_x, tpp, merge_threads, wk.parent);
    } else {
        cc_local_kernel<8><<<local_blocks, kTileW * kTileH, 0, s>>>(bits, g, tiles_x, tpp, wk.parent);
        cc_merge_kernel<8><<<merge_blocks, 256, 0, s>>>(bits, g, tiles_x, tpp, merge_threads, wk.parent);
    }
    cc_flatten_kernel<<<static_cast<unsigned>(seg_blocks), kSegThreads, 0, s>>>(g, wk.parent, wk.seg);
    cc_scan_kernel<<<static_cast<unsigned>(n_planes), 1024, 0, s>>>(g, wk.seg, n_comps);
    cc_number_kernel<<<static_cast<unsigned>(seg_blocks), kSegThreads, 0, s>>>(g, wk.parent, wk.seg, wk);
    cc_stats_kernel<<<static_cast<unsigned>((n_rows + 7) / 8), 256, 0, s>>>(g, static_cast<int>(n_rows), wk.parent,
                                                                            wk, labels);
    cc_select_kernel<<<static_cast<unsigned>(n_planes), 256, 0, s>>>(g, wk, n_comps, max_components, comps);
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        char buf[200];
        snprintf(buf, sizeof buf, "mask_components: launch failed: %s", cudaGetErrorString(e));
        return ub_fail(UNETB200_ECUDA, buf);
    }
    return UNETB200_OK;
}

}  // extern "C"
