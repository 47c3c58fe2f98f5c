// Scoring of predicted mask planes against ground-truth planes (include/unetb200.h, unetb200_mask_match): pixel
// confusion counts and the one-to-one matching of their connected regions at IoU > t, t >= 0.5.  DESIGN.md 6b,
// "Region matching"; oracle/mask_match.py restates it in numpy.
//
// Both stacks are labelled by the union-find of components.cu (cc_label), each into its own components workspace,
// which leaves parent (pixel -> id) and count[id] for every component.  Then, in stream order:
//
//   mt_init_kernel   zeroes the output row of each plane and cand / inter of every pred id
//   mt_vote_kernel   one warp per 8 rows: pixel confusion by ballots; per pred id a, a Boyer-Moore majority vote over the
//                    gt ids (background included) under a's pixels, merged into cand[a] by 64-bit CAS loops
//   mt_inter_kernel  the same walk: inter[a] = |a n cand[a]| exactly
//   mt_match_kernel  one thread per pred id: min_pixels, the IoU test I > t (x) U, the integer sums; cand[a] := I / U
//                    of a matched pair, else 0
//   mt_sum_kernel    one block per plane: iou_sum in a fixed order
//
// Why the candidate is enough: for t >= 0.5 a match means 3I > |a| + |g|, and with I <= |g| that gives 2I > |a|, so a
// partner of a holds a strict majority of a's pixels.  A Boyer-Moore state (value c, count n) stands for n copies of c
// plus pairs of distinct values; merging two states pairs off min(n1, n2) copies of distinct values, so a value with a
// strict majority of the merged pixels is never paired off completely and survives whatever the order of the merges.
// For an `a` without a majority the survivor may depend on scheduling, and the exact test then rejects it.  Every
// output is an integer sum or a function of exact integers, and iou_sum is summed in a fixed order, so the results
// are independent of scheduling.
#include "../../include/unetb200.h"

#include <cuda_runtime.h>

#include <cmath>
#include <cstdio>

#include "cc_internal.h"
#include "errors.h"

namespace {

constexpr int kSumThreads = 256;    // mt_sum_kernel: thread j sums the quotients of ids j, j + 256, ...
constexpr int kRowsPerWarp = 8;     // mt_vote_kernel / mt_inter_kernel: consecutive rows of one plane per warp

// counts[p][k]
enum { kPxTp = 0, kPxFp, kPxFn, kNPred, kNGt, kTp, kSumI, kSumU, kCounts };

// Boyer-Moore state of a pred id: high 32 bits the count, low 32 bits the gt id (-1 = background)
__device__ __forceinline__ unsigned long long bm_state(int g, unsigned n) {
    return (static_cast<unsigned long long>(n) << 32) | static_cast<uint32_t>(g);
}
__device__ __forceinline__ int bm_value(unsigned long long s) { return static_cast<int>(static_cast<uint32_t>(s)); }

__device__ __forceinline__ unsigned long long bm_merge(unsigned long long s, int g, unsigned n) {
    const int c = bm_value(s);
    const unsigned m = static_cast<unsigned>(s >> 32);
    if (c == g) return bm_state(c, m + n);
    return m >= n ? bm_state(c, m - n) : bm_state(g, n - m);
}

struct Match {
    int h, w, cap;
    const int *pp, *pc;               // pred parent / count
    const int *gp, *gc;               // gt parent / count
    const int32_t *np, *ng;           // components per plane
    unsigned long long* cand;         // [P][cap]: Boyer-Moore state, then the quotient bits
    int* inter;                       // [P][cap]
};

// One thread per (plane, id) of the first n_pred[plane] ids; thread 0 of each plane's first block also zeroes the
// plane's counts.
__global__ void __launch_bounds__(256) mt_init_kernel(Match m, int blocks_per_plane, int64_t* __restrict__ counts) {
    const int p = blockIdx.x / blocks_per_plane;
    const int id = (blockIdx.x - p * blocks_per_plane) * 256 + threadIdx.x;
    if (id == 0) {
#pragma unroll
        for (int k = 0; k < kCounts; ++k) counts[static_cast<size_t>(p) * kCounts + k] = 0;
    }
    if (id < m.np[p]) {
        const size_t o = static_cast<size_t>(p) * m.cap + id;
        m.cand[o] = 0;
        m.inter[o] = 0;
    }
}

// Merges the Boyer-Moore state s into *dst with one CAS loop.
__device__ __forceinline__ void bm_merge_into(unsigned long long* dst, unsigned long long s) {
    unsigned long long old = *dst, prev;
    while ((prev = atomicCAS(dst, old, bm_merge(old, bm_value(s), static_cast<unsigned>(s >> 32)))) != old) old = prev;
}

// One warp per kRowsPerWarp consecutive rows of a plane, 32 columns per step.  Lanes with the same (a, g)
// (__match_any_sync) form one group.  The warp carries one pred id `ca` along its rows (the id of the chunk's last
// lane, as a run usually goes on into the next chunk) and merges the groups of `ca` into a local state, flushed into
// cand[ca] with one CAS loop when the carried id changes and at the end; every other group merges into cand[a] from
// its lowest lane.  A region that spans the rows thus costs one CAS per warp instead of one per chunk, which keeps
// the CAS retries on a large region's entry low.
__global__ void __launch_bounds__(256) mt_vote_kernel(Match m, long long n_warps, int64_t* __restrict__ counts) {
    const long long wi = static_cast<long long>(blockIdx.x) * 8 + (threadIdx.x >> 5);
    if (wi >= n_warps) return;                                       // whole warps leave together
    const int wpp = (m.h + kRowsPerWarp - 1) / kRowsPerWarp;
    const int p = static_cast<int>(wi / wpp), y0 = static_cast<int>(wi - static_cast<long long>(p) * wpp) * kRowsPerWarp;
    const int y1 = min(y0 + kRowsPerWarp, m.h);
    const int lane = threadIdx.x & 31;
    const size_t po = static_cast<size_t>(p) * m.h * m.w;
    const int *pp = m.pp + po, *gp = m.gp + po;
    unsigned long long* cand = m.cand + static_cast<size_t>(p) * m.cap;
    long long tp = 0, fp = 0, fn = 0;
    int ca = -1;                                                     // carried pred id (warp-uniform)
    unsigned long long cs = 0;                                       // its local state (warp-uniform)
    for (int y = y0; y < y1; ++y)
    for (int x0 = 0; x0 < m.w; x0 += 32) {
        const int x = x0 + lane;
        int a = -1, g = -1;
        if (x < m.w) {
            a = cc_pixel_id(pp, y * m.w + x);
            g = cc_pixel_id(gp, y * m.w + x);
        }
        const uint32_t bp = __ballot_sync(0xffffffffu, a >= 0), bg = __ballot_sync(0xffffffffu, g >= 0);
        tp += __popc(bp & bg);
        fp += __popc(bp & ~bg);
        fn += __popc(~bp & bg);
        const int a31 = __shfl_sync(0xffffffffu, a, 31);
        if (a31 >= 0 && a31 != ca) {
            if (lane == 0 && ca >= 0 && (cs >> 32)) bm_merge_into(cand + ca, cs);
            ca = a31;
            cs = 0;
        }
        const unsigned long long key = a >= 0 ? bm_state(g, static_cast<unsigned>(a)) : ~0ull;
        const uint32_t grp = __match_any_sync(0xffffffffu, key);
        const bool lead = a >= 0 && lane == __ffs(grp) - 1;
        for (uint32_t mine = __ballot_sync(0xffffffffu, lead && a == ca); mine; mine &= mine - 1) {  // <= 32 rounds
            const int l = __ffs(mine) - 1;
            cs = bm_merge(cs, __shfl_sync(0xffffffffu, g, l), __popc(__shfl_sync(0xffffffffu, grp, l)));
        }
        if (lead && a != ca) bm_merge_into(cand + a, bm_state(g, __popc(grp)));
    }
    if (lane == 0) {
        if (ca >= 0 && (cs >> 32)) bm_merge_into(cand + ca, cs);
        int64_t* c = counts + static_cast<size_t>(p) * kCounts;
        if (tp) atomicAdd(reinterpret_cast<unsigned long long*>(c + kPxTp), static_cast<unsigned long long>(tp));
        if (fp) atomicAdd(reinterpret_cast<unsigned long long*>(c + kPxFp), static_cast<unsigned long long>(fp));
        if (fn) atomicAdd(reinterpret_cast<unsigned long long*>(c + kPxFn), static_cast<unsigned long long>(fn));
    }
}

// Same walk: lanes whose gt id is the candidate of their pred id count towards inter[a]; the carried id's lanes are
// counted in a register (flushed as in mt_vote_kernel), every other group adds its number once from its lowest lane.
__global__ void __launch_bounds__(256) mt_inter_kernel(Match m, long long n_warps) {
    const long long wi = static_cast<long long>(blockIdx.x) * 8 + (threadIdx.x >> 5);
    if (wi >= n_warps) return;
    const int wpp = (m.h + kRowsPerWarp - 1) / kRowsPerWarp;
    const int p = static_cast<int>(wi / wpp), y0 = static_cast<int>(wi - static_cast<long long>(p) * wpp) * kRowsPerWarp;
    const int y1 = min(y0 + kRowsPerWarp, m.h);
    const int lane = threadIdx.x & 31;
    const size_t po = static_cast<size_t>(p) * m.h * m.w;
    const int *pp = m.pp + po, *gp = m.gp + po;
    const unsigned long long* cand = m.cand + static_cast<size_t>(p) * m.cap;
    int* inter = m.inter + static_cast<size_t>(p) * m.cap;
    int ca = -1, cn = 0;                                             // carried pred id and its count (warp-uniform)
    for (int y = y0; y < y1; ++y)
    for (int x0 = 0; x0 < m.w; x0 += 32) {
        const int x = x0 + lane;
        int a = -1;
        if (x < m.w) {
            const int g = cc_pixel_id(gp, y * m.w + x);
            if (g >= 0) {
                a = cc_pixel_id(pp, y * m.w + x);
                if (a >= 0 && bm_value(cand[a]) != g) a = -1;
            }
        }
        const int a31 = __shfl_sync(0xffffffffu, a, 31);
        if (a31 >= 0 && a31 != ca) {
            if (lane == 0 && cn) atomicAdd(inter + ca, cn);
            ca = a31;
            cn = 0;
        }
        cn += __popc(__ballot_sync(0xffffffffu, a >= 0 && a == ca));
        const int other = a != ca ? a : -1;
        const uint32_t grp = __match_any_sync(0xffffffffu, other);
        if (other >= 0 && lane == __ffs(grp) - 1) atomicAdd(inter + other, __popc(grp));
    }
    if (lane == 0 && cn) atomicAdd(inter + ca, cn);
}

__device__ __forceinline__ long long warp_sum(long long v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// One thread per (plane, pred id).  |a| >= min_pixels counts a; a matches cand[a] = g when I > t (x) U, I and U exact
// integers (< 2^31, so exact in fp64) and (x) one correctly rounded fp64 product.  cand[a] becomes the bits of I / U
// for a matched pair, +0.0 otherwise.  Sums are aggregated per warp before the int64 atomics.
__global__ void __launch_bounds__(256) mt_match_kernel(Match m, int blocks_per_plane, int min_pixels, double t,
                                                       int64_t* __restrict__ counts) {
    const int p = blockIdx.x / blocks_per_plane;
    const int id = (blockIdx.x - p * blocks_per_plane) * 256 + threadIdx.x;
    const int n_pred = m.np[p];
    if ((id & ~31) >= n_pred) return;                                // whole warps leave together
    long long kept = 0, tp = 0, si = 0, su = 0;
    if (id < n_pred) {
        const size_t o = static_cast<size_t>(p) * m.cap + id;
        const int na = m.pc[o];
        double q = 0.0;
        if (na >= min_pixels) {
            kept = 1;
            const int g = bm_value(m.cand[o]), in = m.inter[o];
            if (g >= 0 && in > 0) {
                const long long u = static_cast<long long>(na) + m.gc[static_cast<size_t>(p) * m.cap + g] - in;
                if (static_cast<double>(in) > __dmul_rn(t, static_cast<double>(u))) {
                    tp = 1;
                    si = in;
                    su = u;
                    q = __ddiv_rn(static_cast<double>(in), static_cast<double>(u));
                }
            }
        }
        m.cand[o] = static_cast<unsigned long long>(__double_as_longlong(q));
    }
    kept = warp_sum(kept);
    tp = warp_sum(tp);
    si = warp_sum(si);
    su = warp_sum(su);
    if ((threadIdx.x & 31) == 0) {
        auto* c = reinterpret_cast<unsigned long long*>(counts + static_cast<size_t>(p) * kCounts);
        if (kept) atomicAdd(c + kNPred, static_cast<unsigned long long>(kept));
        if (tp) {
            atomicAdd(c + kTp, static_cast<unsigned long long>(tp));
            atomicAdd(c + kSumI, static_cast<unsigned long long>(si));
            atomicAdd(c + kSumU, static_cast<unsigned long long>(su));
        }
    }
}

// One block per plane: thread j adds the quotients of ids j, j + 256, ... in ascending order (starting from +0.0),
// then a fixed pairwise tree (s[j] += s[j + half], half = 128, 64, ..., 1) combines the 256 partial sums.  Writes
// n_gt too.
__global__ void __launch_bounds__(kSumThreads) mt_sum_kernel(Match m, int64_t* __restrict__ counts,
                                                             double* __restrict__ iou_sum) {
    __shared__ double s[kSumThreads];
    const int p = blockIdx.x;
    const int n_pred = m.np[p];
    const unsigned long long* q = m.cand + static_cast<size_t>(p) * m.cap;
    double acc = 0.0;
    for (int id = threadIdx.x; id < n_pred; id += kSumThreads) acc = __dadd_rn(acc, __longlong_as_double(q[id]));
    s[threadIdx.x] = acc;
    __syncthreads();
    for (int half = kSumThreads / 2; half > 0; half >>= 1) {         // 8 rounds
        if (static_cast<int>(threadIdx.x) < half) s[threadIdx.x] = __dadd_rn(s[threadIdx.x], s[threadIdx.x + half]);
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        iou_sum[p] = s[0];
        counts[static_cast<size_t>(p) * kCounts + kNGt] = m.ng[p];
    }
}

// Workspace: pred components workspace, gt components workspace (each rounded up to 16 bytes), cand [P][cap] uint64,
// inter [P][cap] int32, n_comps [2][P] int32.
struct Layout {
    unsigned long long comp, cand, inter, ncomp, total;
};

bool layout_of(int n_planes, int h, int w, Layout* l) {
    const unsigned long long cw = unetb200_components_workspace_bytes(n_planes, h, w);
    if (cw == 0) return false;
    const unsigned long long rows = static_cast<unsigned long long>(n_planes) *
                                    ((static_cast<unsigned long long>(h) * w + 1) / 2);
    l->comp = (cw + 15) & ~15ull;
    l->cand = 2 * l->comp;
    l->inter = l->cand + 8 * rows;
    l->ncomp = l->inter + 4 * rows;
    l->total = l->ncomp + 8ull * n_planes;
    return true;
}

}  // namespace

extern "C" {

uint64_t unetb200_match_workspace_bytes(int n_planes, int h, int w) {
    Layout l;
    if (n_planes <= 0 || !layout_of(n_planes, h, w, &l)) return 0;
    return l.total;
}

int unetb200_mask_match(const uint8_t* pred, int pred_packed, const uint8_t* gt, int gt_packed, int n_planes, int h,
                        int w, int connectivity, int min_pixels, double iou_threshold, int64_t* counts,
                        double* iou_sum, void* workspace, uint64_t workspace_bytes, void* stream) {
    char buf[240];
    auto fail = [&](int code, const char* msg) {
        snprintf(buf, sizeof buf, "mask_match: %s", msg);
        return ub_fail(code, buf);
    };
    Layout l;
    if (!pred || !gt || !counts || !iou_sum || !workspace)
        return fail(UNETB200_EINVAL, "null pointer");
    if ((pred_packed != 0 && pred_packed != 1) || (gt_packed != 0 && gt_packed != 1))
        return fail(UNETB200_EINVAL, "pred_packed and gt_packed must be 0 or 1");
    if (connectivity != 4 && connectivity != 8)
        return fail(UNETB200_EINVAL, "connectivity must be 4 or 8");
    if (min_pixels < 1)
        return fail(UNETB200_EINVAL, "min_pixels must be >= 1");
    if (!std::isfinite(iou_threshold) || iou_threshold < 0.5 || iou_threshold >= 1.0)
        return fail(UNETB200_EINVAL, "iou_threshold must be in [0.5, 1)");
    if (n_planes <= 0 || !layout_of(n_planes, h, w, &l))
        return fail(UNETB200_EINVAL, "bad size (n_planes, h, w >= 1 and h * w < 2^31)");
    if ((pred_packed || gt_packed) && (w & 31))
        return fail(UNETB200_EINVAL, "bit-packed planes need w % 32 == 0");
    if (((pred_packed ? reinterpret_cast<uintptr_t>(pred) : 0) | (gt_packed ? reinterpret_cast<uintptr_t>(gt) : 0)) & 3 ||
        ((reinterpret_cast<uintptr_t>(counts) | reinterpret_cast<uintptr_t>(iou_sum)) & 7) ||
        (reinterpret_cast<uintptr_t>(workspace) & 15))
        return fail(UNETB200_EINVAL, "misaligned pointer (bit-packed planes 4-byte aligned, counts and iou_sum 8-byte "
                                     "aligned, workspace 16-byte aligned)");
    if (workspace_bytes < l.total)
        return fail(UNETB200_ENOMEM, "workspace smaller than unetb200_match_workspace_bytes");
    const int blocks_per_plane = static_cast<int>(((static_cast<long long>(h) * w + 1) / 2 + 255) / 256);
    if (!cc_batch_fits(n_planes, h, w) || static_cast<long long>(blocks_per_plane) * n_planes >= (1LL << 31))
        return fail(UNETB200_EINVAL, "batch too large");

    cudaStream_t s = static_cast<cudaStream_t>(stream);
    char* ws = static_cast<char*>(workspace);
    auto* ncomp = reinterpret_cast<int32_t*>(ws + l.ncomp);
    CcLabels lp, lg;
    int rc = cc_label("mask_match", pred, pred_packed, n_planes, h, w, connectivity, ws, ncomp, s, &lp);
    if (rc != UNETB200_OK) return rc;
    rc = cc_label("mask_match", gt, gt_packed, n_planes, h, w, connectivity, ws + l.comp, ncomp + n_planes, s, &lg);
    if (rc != UNETB200_OK) return rc;
    Match m;
    m.h = h;
    m.w = w;
    m.cap = lp.cap;
    m.pp = lp.parent;
    m.pc = lp.count;
    m.gp = lg.parent;
    m.gc = lg.count;
    m.np = ncomp;
    m.ng = ncomp + n_planes;
    m.cand = reinterpret_cast<unsigned long long*>(ws + l.cand);
    m.inter = reinterpret_cast<int*>(ws + l.inter);
    const unsigned id_blocks = static_cast<unsigned>(static_cast<long long>(blocks_per_plane) * n_planes);
    const long long n_warps = static_cast<long long>(n_planes) * ((h + kRowsPerWarp - 1) / kRowsPerWarp);
    const unsigned row_blocks = static_cast<unsigned>((n_warps + 7) / 8);
    mt_init_kernel<<<id_blocks, 256, 0, s>>>(m, blocks_per_plane, counts);
    mt_vote_kernel<<<row_blocks, 256, 0, s>>>(m, n_warps, counts);
    mt_inter_kernel<<<row_blocks, 256, 0, s>>>(m, n_warps);
    mt_match_kernel<<<id_blocks, 256, 0, s>>>(m, blocks_per_plane, min_pixels, iou_threshold, counts);
    mt_sum_kernel<<<static_cast<unsigned>(n_planes), kSumThreads, 0, s>>>(m, counts, iou_sum);
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        snprintf(buf, sizeof buf, "mask_match: launch failed: %s", cudaGetErrorString(e));
        return ub_fail(UNETB200_ECUDA, buf);
    }
    return UNETB200_OK;
}

}  // extern "C"
