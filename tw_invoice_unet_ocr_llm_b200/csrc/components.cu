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
//
// unetb200_mask_components_oriented runs the same passes, then the oriented-box passes of the selected components
// (cc_moments_kernel ... cc_obox_kernel, below).  Their floating-point results are min / max of values that do not
// depend on the order of work, so they are deterministic too.
//
// cc_fill_holes (unetb200_mask_morph, op UNETB200_MORPH_FILL_HOLES) labels the complement of the planes with the
// same union-find: cc_pack_kernel in a complement mode, cc_local / cc_merge (4-connectivity) and cc_flatten, then
// cc_border_kernel marks the roots of the components that reach the border and cc_fill_kernel writes the planes
// with every unmarked background component set.
//
// cc_label (unetb200_mask_match, csrc/match.cu) runs the passes pack .. stats without the selection, so the
// workspace keeps the pixel -> component map and the size of every component of a plane.
#include "../../include/unetb200.h"

#include <cuda_runtime.h>

#include <climits>
#include <cstdio>

#include "cc_internal.h"
#include "errors.h"

namespace {

constexpr int kTileW = 32, kTileH = 16;        // cc_local_kernel: one thread per pixel of a tile
constexpr int kSeg = 1024;                     // raster pixels per root-count segment
constexpr int kSegThreads = 256;
constexpr int kMaxK = 16;
constexpr int kBg = -1;                        // parent entry of a background pixel
constexpr int kBorderRoot = -2;                // cc_fill_holes: parent entry of a root whose component reaches the border

// What cc_pack_kernel sets a bit for
enum PackMode { kPackSet = 0 /* a non-zero byte */, kPackClearBytes = 1 /* a zero byte */,
                kPackClearBits = 2 /* a clear bit of bit-packed planes with w % 32 == 0 */ };

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
                                                      int mode, uint32_t* __restrict__ bits) {
    const long long t = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    const long long word = t >> 5;                       // one warp per word, one lane per pixel
    if (word >= static_cast<long long>(n_planes) * g.wpp) return;     // whole warps leave together
    if (mode == kPackClearBits) {                        // same layout, no pad bits: the complement is ~word
        if ((threadIdx.x & 31) == 0) bits[word] = ~__ldg(reinterpret_cast<const uint32_t*>(mask) + word);
        return;
    }
    const int p = static_cast<int>(word / g.wpp), wi = static_cast<int>(word - static_cast<long long>(p) * g.wpp);
    const int i = (wi << 5) + static_cast<int>(threadIdx.x & 31);
    const bool on = i < g.n && (mask[static_cast<size_t>(p) * g.n + i] != 0) == (mode == kPackSet);
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

Work work_of(void* workspace, int n_planes, const Plane& g) {
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
    return wk;
}

// Grid sizes of the labelling passes; false when one of them reaches 2^31 blocks or threads.
struct Grids {
    int tiles_x, tiles_per_plane;
    long long merge_threads, seg_blocks, pack_blocks;
};
bool grids_of(int n_planes, const Plane& g, Grids* gr) {
    gr->tiles_x = (g.w + kTileW - 1) / kTileW;
    const long long tiles = static_cast<long long>(gr->tiles_x) * ((g.h + kTileH - 1) / kTileH);
    gr->tiles_per_plane = static_cast<int>(tiles);
    gr->merge_threads = tiles * n_planes * 64;
    gr->seg_blocks = static_cast<long long>(n_planes) * g.nseg;
    gr->pack_blocks = (static_cast<long long>(n_planes) * g.wpp * 32 + 255) / 256;
    return tiles * n_planes < (1LL << 31) && static_cast<long long>(n_planes) * g.h < (1LL << 31) &&
           gr->seg_blocks < (1LL << 31) && gr->pack_blocks < (1LL << 31);
}

// The labelling passes pack .. stats: afterwards parent[i] names the component of pixel i (cc_pixel_id),
// count[id] is the size of every component and n_comps[plane] their number.  Sizes already validated, grids
// checked by grids_of.
void label_passes(const uint8_t* mask, int packed, int n_planes, const Plane& g, const Grids& gr, int connectivity,
                  const Work& wk, int32_t* labels, int32_t* n_comps, cudaStream_t s) {
    const int tiles_x = gr.tiles_x;
    const long long n_rows = static_cast<long long>(n_planes) * g.h;
    const long long seg_blocks = gr.seg_blocks;
    const uint32_t* bits = wk.bits;
    if (packed) {
        bits = reinterpret_cast<const uint32_t*>(mask);  // [h][w/8] with w % 32 == 0 is the plane-contiguous layout
    } else {
        cc_pack_kernel<<<static_cast<unsigned>(gr.pack_blocks), 256, 0, s>>>(mask, n_planes, g, kPackSet, wk.bits);
    }
    const int tpp = gr.tiles_per_plane;
    const unsigned local_blocks = static_cast<unsigned>(static_cast<long long>(tpp) * n_planes);
    const long long merge_threads = gr.merge_threads;
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
}

// ---------------------------------------------------------------- hole filling (cc_fill_holes)
// After cc_flatten_kernel over the complement, parent[i] is the root of background pixel i (kBg: a set pixel).
// One thread per (plane, border position): the root of a background border pixel becomes kBorderRoot.  Only root
// entries are written, all with the same value, and a non-root entry still names its root, so the order of the
// writes does not matter.  Corner pixels come twice, which is harmless.
__global__ void __launch_bounds__(256) cc_border_kernel(Plane g, long long n_threads, int* __restrict__ parent) {
    const long long t = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (t >= n_threads) return;
    const long long per = 2LL * (g.w + g.h), w = g.w;
    const int p = static_cast<int>(t / per);
    const long long k = t - p * per;
    int x, y;
    if (k < w) { x = static_cast<int>(k); y = 0; }
    else if (k < 2 * w) { x = static_cast<int>(k - w); y = g.h - 1; }
    else if (k < 2 * w + g.h) { x = 0; y = static_cast<int>(k - 2 * w); }
    else { x = g.w - 1; y = static_cast<int>(k - 2 * w - g.h); }
    int* par = parent + static_cast<size_t>(p) * g.n;
    const int v = par[y * g.w + x];
    if (v != kBg && v != kBorderRoot) par[v] = kBorderRoot;
}

// One warp per 32-pixel word (as cc_pack_kernel): a pixel is set when it is set in the input (kBg) or its
// background component has an unmarked root.  Bit-packed output (w % 32 == 0) has the plane-contiguous word layout.
__global__ void __launch_bounds__(256) cc_fill_kernel(Plane g, int n_planes, const int* __restrict__ parent,
                                                      int out_packed, uint8_t* __restrict__ out) {
    const long long t = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    const long long word = t >> 5;
    if (word >= static_cast<long long>(n_planes) * g.wpp) return;     // whole warps leave together
    const int p = static_cast<int>(word / g.wpp), wi = static_cast<int>(word - static_cast<long long>(p) * g.wpp);
    const int i = (wi << 5) + static_cast<int>(threadIdx.x & 31);
    const int* par = parent + static_cast<size_t>(p) * g.n;
    bool on = false;
    if (i < g.n) {
        const int v = par[i];
        on = v == kBg || (v != kBorderRoot && par[v] != kBorderRoot);
    }
    if (out_packed) {
        const uint32_t b = __ballot_sync(0xffffffffu, on);
        if ((threadIdx.x & 31) == 0) reinterpret_cast<uint32_t*>(out)[word] = b;
    } else if (i < g.n) {
        out[static_cast<size_t>(p) * g.n + i] = on ? 1 : 0;
    }
}

// ---------------------------------------------------------------- oriented boxes of the selected components
// (unetb200_mask_components_oriented): three more passes over the parent array after cc_select_kernel.
//
//   cc_moments_kernel  raw moments n, Sx, Sy, Sxx, Sxy, Syy of each selected component (int64 atomics)
//   cc_axis_kernel     principal axis e1 of each selected row from its moments and the plane's frame scale
//   cc_extent_kernel   min / max of the projections u = P.e1, v = P.e2 of the component's frame points P
//   cc_obox_kernel     extents back to float64 (unused rows: zeros)
//
// The geometry uses integer arithmetic and correctly rounded fp64 + - * / sqrt only (__d*_rn: no FMA contraction,
// no transcendental function), so oracle/oriented.py restates it bit for bit.
constexpr int kMaxSide = 32767;      // h, w <= 32767: n * w^2 < 2^61, every moment sum is exact in int64

// Workspace tail of the oriented call, behind the components workspace (16-byte aligned): [P][kMaxK][4] int64 =
// order-preserving images of umin, umax, vmin, vmax.
unsigned long long oriented_tail_offset(int n_planes, const Plane& g) {
    return (4ull * work_words(n_planes, g) + 15ull) & ~15ull;
}
unsigned long long oriented_bytes(int n_planes, const Plane& g) {
    return oriented_tail_offset(n_planes, g) + static_cast<unsigned long long>(n_planes) * kMaxK * 4 * 8;
}

// Row of the plane's selection that holds component `id`, or -1 (ids are unique within a plane).
__device__ __forceinline__ int slot_of(const int* sel, int k_out, int id) {
    int s = -1;
    if (id >= 0) {
        for (int k = 0; k < k_out; ++k) s = sel[k] == id ? k : s;
    }
    return s;
}

// sel[k] = id of the plane's k-th selected component (comps[..., 5] - 1; -1 for an unused row)
__device__ __forceinline__ void load_selection(const int32_t* __restrict__ comps, int p, int k_out, int* sel) {
    if (threadIdx.x < kMaxK)
        sel[threadIdx.x] = static_cast<int>(threadIdx.x) < k_out
                               ? comps[(static_cast<size_t>(p) * k_out + threadIdx.x) * 6 + 5] - 1 : -1;
}

// Order-preserving int64 image of a double (signed compare of the images == numeric compare; -0 < +0) and back.
__device__ __forceinline__ long long dkey(double d) {
    const long long b = __double_as_longlong(d);
    return b >= 0 ? b : b ^ 0x7fffffffffffffffLL;
}
__device__ __forceinline__ double dkey_inv(long long k) {
    return __longlong_as_double(k >= 0 ? k : k ^ 0x7fffffffffffffffLL);
}

// One warp per row (blockIdx.y = plane, 8 rows per block), 32 columns per step.  Lanes of the same selected
// component (__match_any_sync) add their pixels with one set of atomics from the lowest lane: the group's lanes l
// lie in one row y at x = x0 + l, so with c = popc, S1 = sum l and S2 = sum l^2 (bit sums of the group mask)
// Sx = c x0 + S1, Sxx = c x0^2 + 2 x0 S1 + S2, Sy = c y, Sxy = y Sx, Syy = c y^2.
__global__ void __launch_bounds__(256) cc_moments_kernel(Plane g, const int* __restrict__ parent,
                                                         const int32_t* __restrict__ comps, int k_out,
                                                         unsigned long long* __restrict__ mom) {
    __shared__ int sel[kMaxK];
    const int p = blockIdx.y;
    load_selection(comps, p, k_out, sel);
    __syncthreads();
    const int y = blockIdx.x * 8 + static_cast<int>(threadIdx.x >> 5);
    if (y >= g.h) return;                                            // whole warps leave together
    const int lane = threadIdx.x & 31;
    const int* par = parent + static_cast<size_t>(p) * g.n;
    unsigned long long* mp = mom + static_cast<size_t>(p) * k_out * 6;
    const uint32_t bit[5] = {0xaaaaaaaau, 0xccccccccu, 0xf0f0f0f0u, 0xff00ff00u, 0xffff0000u};   // bit j of lane index
    for (int x0 = 0; x0 < g.w; x0 += 32) {
        const int x = x0 + lane;
        const int slot = x < g.w ? slot_of(sel, k_out, cc_pixel_id(par, y * g.w + x)) : -1;
        const uint32_t grp = __match_any_sync(0xffffffffu, slot);
        if (slot >= 0 && lane == __ffs(grp) - 1) {
            long long s1 = 0, s2 = 0;
#pragma unroll
            for (int j = 0; j < 5; ++j) {
                s1 += static_cast<long long>(__popc(grp & bit[j])) << j;
#pragma unroll
                for (int k = 0; k < 5; ++k) s2 += static_cast<long long>(__popc(grp & bit[j] & bit[k])) << (j + k);
            }
            const long long c = __popc(grp), X0 = x0, Y = y;
            const long long sx = c * X0 + s1;
            unsigned long long* o = mp + slot * 6;
            atomicAdd(o + 0, static_cast<unsigned long long>(c));
            atomicAdd(o + 1, static_cast<unsigned long long>(sx));
            atomicAdd(o + 2, static_cast<unsigned long long>(c * Y));
            atomicAdd(o + 3, static_cast<unsigned long long>(c * X0 * X0 + 2 * X0 * s1 + s2));
            atomicAdd(o + 4, static_cast<unsigned long long>(sx * Y));
            atomicAdd(o + 5, static_cast<unsigned long long>(c * Y * Y));
        }
    }
}

// Signed 128-bit integer -> fp64, rounded to nearest-even (as Python's float(int)): values below 2^63 go through
// __ull2double_rn; larger ones are cut to their top 63 bits with a sticky bit for what was cut (it lies below the
// rounding position of a 53-bit significand), converted, and scaled back by an exact power of two.
__device__ __forceinline__ double i128_to_double_rn(__int128 v) {
    const bool neg = v < 0;
    const unsigned __int128 m = neg ? -static_cast<unsigned __int128>(v) : static_cast<unsigned __int128>(v);
    double d;
    if ((m >> 63) == 0) {
        d = __ull2double_rn(static_cast<unsigned long long>(m));
    } else {
        const unsigned long long hi = static_cast<unsigned long long>(m >> 64);
        const int s = (hi ? 128 - __clzll(static_cast<long long>(hi)) : 64) - 63;      // 1 .. 65
        unsigned long long t = static_cast<unsigned long long>(m >> s);
        if (m & ((static_cast<unsigned __int128>(1) << s) - 1)) t |= 1ull;
        d = __dmul_rn(__ull2double_rn(t), __longlong_as_double(static_cast<long long>(1023 + s) << 52));
    }
    return neg ? -d : d;
}

// One thread per (plane, row): e1 of DESIGN 6b from the exact covariances; initialises the extent keys.
__global__ void __launch_bounds__(256) cc_axis_kernel(int n_rows, int k_out, const double* __restrict__ scale,
                                                      const long long* __restrict__ mom, double* __restrict__ obox,
                                                      long long* __restrict__ keys) {
    const int r = blockIdx.x * 256 + threadIdx.x;
    if (r >= n_rows) return;
    const int p = r / k_out;
    const long long* m = mom + static_cast<size_t>(r) * 6;
    long long* kr = keys + static_cast<size_t>(r) * 4;
    kr[0] = LLONG_MAX; kr[1] = LLONG_MIN; kr[2] = LLONG_MAX; kr[3] = LLONG_MIN;
    double ex = 0.0, ey = 0.0;
    const long long n = m[0];
    if (n > 0) {
        const double sx = scale ? scale[2 * p] : 1.0, sy = scale ? scale[2 * p + 1] : 1.0;
        const __int128 N = n, Sx = m[1], Sy = m[2];
        const double cxx = i128_to_double_rn(N * m[3] - Sx * Sx);
        const double cxy = i128_to_double_rn(N * m[4] - Sx * Sy);
        const double cyy = i128_to_double_rn(N * m[5] - Sy * Sy);
        const double a = __dmul_rn(__dmul_rn(sx, sx), cxx);
        const double b = __dmul_rn(__dmul_rn(sx, sy), cxy);
        const double c = __dmul_rn(__dmul_rn(sy, sy), cyy);
        if (b == 0.0) {
            ex = a >= c ? 1.0 : 0.0;
            ey = a >= c ? 0.0 : 1.0;
        } else {
            const double amc = __dadd_rn(a, -c);
            const double d = __dsqrt_rn(__dadd_rn(__dmul_rn(amc, amc), __dmul_rn(4.0, __dmul_rn(b, b))));
            double vx, vy;
            if (a >= c) {
                vx = __dadd_rn(amc, d);
                vy = __dmul_rn(2.0, b);
            } else {
                vx = __dmul_rn(2.0, b);
                vy = __dadd_rn(__dadd_rn(c, -a), d);
            }
            const double nrm = __dsqrt_rn(__dadd_rn(__dmul_rn(vx, vx), __dmul_rn(vy, vy)));
            ex = __ddiv_rn(vx, nrm);
            ey = __ddiv_rn(vy, nrm);
            if (ex < 0.0 || (ex == 0.0 && ey < 0.0)) {
                ex = -ex;
                ey = -ey;
            }
        }
    }
    obox[static_cast<size_t>(r) * 6 + 0] = ex;
    obox[static_cast<size_t>(r) * 6 + 1] = ey;
}

// Frame point of a mask pixel and its projections u = X e1x + Y e1y, v = X e2x + Y e2y (e2 = (-e1y, e1x)).
__device__ __forceinline__ void project(int x, int y, double sx, double sy, double ex, double ey, double& u,
                                        double& v) {
    const double X = __dadd_rn(__dmul_rn(__dadd_rn(static_cast<double>(x), 0.5), sx), -0.5);
    const double Y = __dadd_rn(__dmul_rn(__dadd_rn(static_cast<double>(y), 0.5), sy), -0.5);
    u = __dadd_rn(__dmul_rn(X, ex), __dmul_rn(Y, ey));
    v = __dadd_rn(__dmul_rn(X, -ey), __dmul_rn(Y, ex));
}

// Same walk as cc_moments_kernel.  Within a row, X grows with x, Y is fixed, and a correctly rounded product with
// a fixed factor and a correctly rounded sum with a fixed term are monotone: u and v are monotone in x along the
// row, so a group's extremes are at its first and last lane and the lowest lane projects just those two pixels.
__global__ void __launch_bounds__(256) cc_extent_kernel(Plane g, const int* __restrict__ parent,
                                                        const int32_t* __restrict__ comps, int k_out,
                                                        const double* __restrict__ scale,
                                                        const double* __restrict__ obox, long long* __restrict__ keys) {
    __shared__ int sel[kMaxK];
    __shared__ double e1[kMaxK][2];
    const int p = blockIdx.y;
    load_selection(comps, p, k_out, sel);
    if (threadIdx.x < static_cast<unsigned>(2 * k_out))
        e1[threadIdx.x >> 1][threadIdx.x & 1] = obox[(static_cast<size_t>(p) * k_out + (threadIdx.x >> 1)) * 6 + (threadIdx.x & 1)];
    __syncthreads();
    const int y = blockIdx.x * 8 + static_cast<int>(threadIdx.x >> 5);
    if (y >= g.h) return;
    const int lane = threadIdx.x & 31;
    const double sx = scale ? scale[2 * p] : 1.0, sy = scale ? scale[2 * p + 1] : 1.0;
    const int* par = parent + static_cast<size_t>(p) * g.n;
    long long* kp = keys + static_cast<size_t>(p) * k_out * 4;
    for (int x0 = 0; x0 < g.w; x0 += 32) {
        const int x = x0 + lane;
        const int slot = x < g.w ? slot_of(sel, k_out, cc_pixel_id(par, y * g.w + x)) : -1;
        const uint32_t grp = __match_any_sync(0xffffffffu, slot);
        if (slot >= 0 && lane == __ffs(grp) - 1) {
            double u0, v0, u1, v1;
            project(x, y, sx, sy, e1[slot][0], e1[slot][1], u0, v0);
            project(x0 + 31 - __clz(grp), y, sx, sy, e1[slot][0], e1[slot][1], u1, v1);
            long long* o = kp + slot * 4;
            atomicMin(o + 0, min(dkey(u0), dkey(u1)));
            atomicMax(o + 1, max(dkey(u0), dkey(u1)));
            atomicMin(o + 2, min(dkey(v0), dkey(v1)));
            atomicMax(o + 3, max(dkey(v0), dkey(v1)));
        }
    }
}

// One thread per (plane, row): obox[2..5] = the extents (rows without pixels: zeros).
__global__ void __launch_bounds__(256) cc_obox_kernel(int n_rows, const long long* __restrict__ mom,
                                                      const long long* __restrict__ keys, double* __restrict__ obox) {
    const int r = blockIdx.x * 256 + threadIdx.x;
    if (r >= n_rows) return;
    const bool live = mom[static_cast<size_t>(r) * 6] > 0;
#pragma unroll
    for (int j = 0; j < 4; ++j)
        obox[static_cast<size_t>(r) * 6 + 2 + j] = live ? dkey_inv(keys[static_cast<size_t>(r) * 4 + j]) : 0.0;
}

// Outputs of the oriented call (null for unetb200_mask_components)
struct OrientedOut {
    const double* scale;
    int64_t* moments;
    double* obox;
};

// Body of both entry points: validation (every failure before any CUDA call), then the labelling passes and,
// with `ori`, the oriented passes.  `who` prefixes the error messages.
int components_impl(const char* who, const uint8_t* mask, int packed, int n_planes, int h, int w, int connectivity,
                    int max_components, int32_t* labels, int32_t* comps, int32_t* n_comps, void* workspace,
                    uint64_t workspace_bytes, void* stream, const OrientedOut* ori) {
    char buf[240];
    auto fail = [&](int code, const char* msg) {
        snprintf(buf, sizeof buf, "%s: %s", who, msg);
        return ub_fail(code, buf);
    };
    Plane g;
    if (!mask || !comps || !n_comps || !workspace)
        return fail(UNETB200_EINVAL, "null pointer");
    if (connectivity != 4 && connectivity != 8)
        return fail(UNETB200_EINVAL, "connectivity must be 4 or 8");
    if (max_components < 1 || max_components > kMaxK)
        return fail(UNETB200_EINVAL, "max_components must be in [1, 16]");
    if (packed != 0 && packed != 1)
        return fail(UNETB200_EINVAL, "packed must be 0 or 1");
    if (n_planes <= 0 || !plane_of(h, w, &g))
        return fail(UNETB200_EINVAL, "bad size (n_planes, h, w >= 1 and h * w < 2^31)");
    if (packed && (w & 31))
        return fail(UNETB200_EINVAL, "bit-packed planes need w % 32 == 0");
    if (((packed ? reinterpret_cast<uintptr_t>(mask) : 0) | reinterpret_cast<uintptr_t>(labels) |
         reinterpret_cast<uintptr_t>(comps) | reinterpret_cast<uintptr_t>(n_comps)) & 3 ||
        (reinterpret_cast<uintptr_t>(workspace) & 15))
        return fail(UNETB200_EINVAL, "misaligned pointer (int32 outputs and bit-packed planes "
                                     "4-byte aligned, workspace 16-byte aligned)");
    if (ori) {
        if (!ori->moments || !ori->obox)
            return fail(UNETB200_EINVAL, "null pointer");
        if ((reinterpret_cast<uintptr_t>(ori->moments) | reinterpret_cast<uintptr_t>(ori->obox) |
             reinterpret_cast<uintptr_t>(ori->scale)) & 7)
            return fail(UNETB200_EINVAL, "misaligned pointer (moments, obox and scale 8-byte aligned)");
        if (h > kMaxSide || w > kMaxSide)
            return fail(UNETB200_EINVAL, "planes larger than 32767 pixels on a side");
        if (n_planes > 65535)
            return fail(UNETB200_EINVAL, "batch too large (at most 65535 planes)");
        if (workspace_bytes < oriented_bytes(n_planes, g))
            return fail(UNETB200_ENOMEM, "workspace smaller than unetb200_components_oriented_workspace_bytes");
    } else if (workspace_bytes < 4ull * work_words(n_planes, g)) {
        return fail(UNETB200_ENOMEM, "workspace smaller than unetb200_components_workspace_bytes");
    }
    Grids gr;
    if (!grids_of(n_planes, g, &gr))
        return fail(UNETB200_EINVAL, "batch too large");
    const Work wk = work_of(workspace, n_planes, g);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    label_passes(mask, packed, n_planes, g, gr, connectivity, wk, labels, n_comps, s);
    cc_select_kernel<<<static_cast<unsigned>(n_planes), 256, 0, s>>>(g, wk, n_comps, max_components, comps);
    if (ori) {
        const int k = max_components, rows = n_planes * k;
        long long* keys = reinterpret_cast<long long*>(static_cast<char*>(workspace) + oriented_tail_offset(n_planes, g));
        const dim3 walk(static_cast<unsigned>((h + 7) / 8), static_cast<unsigned>(n_planes));
        const unsigned row_blocks = static_cast<unsigned>((rows + 255) / 256);
        cudaError_t e = cudaMemsetAsync(ori->moments, 0, static_cast<size_t>(rows) * 6 * sizeof(int64_t), s);
        if (e != cudaSuccess) {
            snprintf(buf, sizeof buf, "%s: memset failed: %s", who, cudaGetErrorString(e));
            return ub_fail(UNETB200_ECUDA, buf);
        }
        auto* mom = reinterpret_cast<unsigned long long*>(ori->moments);
        const auto* smom = reinterpret_cast<const long long*>(ori->moments);
        cc_moments_kernel<<<walk, 256, 0, s>>>(g, wk.parent, comps, k, mom);
        cc_axis_kernel<<<row_blocks, 256, 0, s>>>(rows, k, ori->scale, smom, ori->obox, keys);
        cc_extent_kernel<<<walk, 256, 0, s>>>(g, wk.parent, comps, k, ori->scale, ori->obox, keys);
        cc_obox_kernel<<<row_blocks, 256, 0, s>>>(rows, smom, keys, ori->obox);
    }
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        snprintf(buf, sizeof buf, "%s: launch failed: %s", who, cudaGetErrorString(e));
        return ub_fail(UNETB200_ECUDA, buf);
    }
    return UNETB200_OK;
}

}  // namespace

int cc_fill_holes(const char* who, const uint8_t* in, int in_packed, uint8_t* out, int out_packed, int n_planes,
                  int h, int w, void* workspace, cudaStream_t s) {
    char buf[240];
    Plane g;
    Grids gr;
    plane_of(h, w, &g);
    const long long border_threads = static_cast<long long>(n_planes) * 2 * (static_cast<long long>(w) + h);
    if (!grids_of(n_planes, g, &gr) || (border_threads + 255) / 256 >= (1LL << 31)) {
        snprintf(buf, sizeof buf, "%s: batch too large", who);
        return ub_fail(UNETB200_EINVAL, buf);
    }
    const Work wk = work_of(workspace, n_planes, g);
    const unsigned pack_blocks = static_cast<unsigned>(gr.pack_blocks);
    const unsigned local_blocks = static_cast<unsigned>(static_cast<long long>(gr.tiles_per_plane) * n_planes);
    const unsigned merge_blocks = static_cast<unsigned>((gr.merge_threads + 255) / 256);
    cc_pack_kernel<<<pack_blocks, 256, 0, s>>>(in, n_planes, g, in_packed ? kPackClearBits : kPackClearBytes,
                                               wk.bits);
    cc_local_kernel<4><<<local_blocks, kTileW * kTileH, 0, s>>>(wk.bits, g, gr.tiles_x, gr.tiles_per_plane,
                                                                wk.parent);
    cc_merge_kernel<4><<<merge_blocks, 256, 0, s>>>(wk.bits, g, gr.tiles_x, gr.tiles_per_plane, gr.merge_threads,
                                                    wk.parent);
    cc_flatten_kernel<<<static_cast<unsigned>(gr.seg_blocks), kSegThreads, 0, s>>>(g, wk.parent, wk.seg);
    cc_border_kernel<<<static_cast<unsigned>((border_threads + 255) / 256), 256, 0, s>>>(g, border_threads,
                                                                                        wk.parent);
    cc_fill_kernel<<<pack_blocks, 256, 0, s>>>(g, n_planes, wk.parent, out_packed, out);
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        snprintf(buf, sizeof buf, "%s: launch failed: %s", who, cudaGetErrorString(e));
        return ub_fail(UNETB200_ECUDA, buf);
    }
    return UNETB200_OK;
}

bool cc_batch_fits(int n_planes, int h, int w) {
    Plane g;
    Grids gr;
    return n_planes > 0 && plane_of(h, w, &g) && grids_of(n_planes, g, &gr);
}

int cc_label(const char* who, const uint8_t* mask, int packed, int n_planes, int h, int w, int connectivity,
             void* workspace, int32_t* n_comps, cudaStream_t s, CcLabels* out) {
    char buf[240];
    Plane g;
    Grids gr;
    if (n_planes <= 0 || !plane_of(h, w, &g) || !grids_of(n_planes, g, &gr)) {
        snprintf(buf, sizeof buf, "%s: batch too large", who);
        return ub_fail(UNETB200_EINVAL, buf);
    }
    const Work wk = work_of(workspace, n_planes, g);
    label_passes(mask, packed, n_planes, g, gr, connectivity, wk, nullptr, n_comps, s);
    out->parent = wk.parent;
    out->count = wk.count;
    out->cap = g.cap;
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        snprintf(buf, sizeof buf, "%s: launch failed: %s", who, cudaGetErrorString(e));
        return ub_fail(UNETB200_ECUDA, buf);
    }
    return UNETB200_OK;
}

extern "C" {

uint64_t unetb200_components_workspace_bytes(int n_planes, int h, int w) {
    Plane g;
    if (n_planes <= 0 || !plane_of(h, w, &g)) return 0;
    return 4ull * work_words(n_planes, g);
}

uint64_t unetb200_components_oriented_workspace_bytes(int n_planes, int h, int w) {
    Plane g;
    if (n_planes <= 0 || n_planes > 65535 || h > kMaxSide || w > kMaxSide || !plane_of(h, w, &g)) return 0;
    return oriented_bytes(n_planes, g);
}

int unetb200_mask_components(const uint8_t* mask, int packed, int n_planes, int h, int w, int connectivity,
                             int max_components, int32_t* labels, int32_t* comps, int32_t* n_comps, void* workspace,
                             uint64_t workspace_bytes, void* stream) {
    return components_impl("mask_components", mask, packed, n_planes, h, w, connectivity, max_components, labels,
                           comps, n_comps, workspace, workspace_bytes, stream, nullptr);
}

int unetb200_mask_components_oriented(const uint8_t* mask, int packed, int n_planes, int h, int w, int connectivity,
                                      int max_components, const double* scale, int32_t* labels, int32_t* comps,
                                      int32_t* n_comps, int64_t* moments, double* obox, void* workspace,
                                      uint64_t workspace_bytes, void* stream) {
    const OrientedOut ori{scale, moments, obox};
    return components_impl("mask_components_oriented", mask, packed, n_planes, h, w, connectivity, max_components,
                           labels, comps, n_comps, workspace, workspace_bytes, stream, &ori);
}

}  // extern "C"
