// Implicit-GEMM convolution on the sm_100a tensor cores (tcgen05 + TMEM + TMA).
//
// One kernel template covers every dense contraction of the U-Net forward
// (reference: unet_model.py:9-17 DoubleConv convs, :38-47 ConvTranspose2d):
//
//   TAPS == 9 : 3x3 / pad 1 / stride 1 convolution, NHWC bf16 activations,
//               weights packed [tap][Cout][Cin] bf16 with BatchNorm folded in.
//               Up to two activation sources are read back to back along K,
//               which is torch.cat([up, skip], dim=1) without the copy
//               (unet_model.py:71,75,79,83).
//   TAPS == 1 : ConvTranspose2d(k=2, s=2) as one GEMM with N = 4*Cout
//               (rows of B ordered [tap = 2a+b][Cout]); the epilogue scatters
//               column block `tap` to output pixel (2y+a, 2x+b).
//
// GEMM view: D[M=128 pixels (16 rows x 8 cols of one image), N=BN channels]
//            += A[128, 64] * B[BN, 64]^T  per (channel slice of 64, tap).
//
// How the A operand (activations) reaches shared memory -- `AMODE`:
//   A_TAP   : one 16x8 TMA box per (slice, tap), shifted by the tap offset.
//             Fully standard SWIZZLE_128B K-major tile; 9x the smem fill traffic.
//   A_COL3  : one 18x8 box per (slice, kx): the three ky taps of that column
//             shift are the same patch read 0/1/2 rows (= 1024 B, a whole
//             swizzle atom) further down, so the layout stays canonical.
//             3.4x the fill traffic of one tile.
//   A_HALO  : one 18x10 box per slice; the nine taps are nine descriptors into
//             it, start address shifted by (ky*10+kx) rows of 128 B and the
//             8-row group stride set to one patch row (1280 B).  1.4x traffic,
//             but relies on the swizzle being a function of the absolute smem
//             address (validated on hardware by tests/test_conv_kernels.py).
// TMA zero-fills out-of-bounds box elements, which is the conv zero padding.
//   A_STEM  : first conv of the network (Cin = n_channels <= 3, K = 9*Cin <= 27): eight extra
//             warps (two groups of 128 threads taking alternate tiles) build the im2col rows
//             themselves, straight from the user's fp32 NCHW / uint8 NHWC tensor, as bf16
//             hi | lo halves of one 64-wide K slice (x = hi + lo to 16 significand bits); the GEMM
//             is [x_hi | x_lo] * [w_hi | w_hi] + x_hi * w_lo, i.e. fp32-class accuracy from bf16
//             MMAs.  The layer is HBM-bound (64 bf16 channels out per pixel); the MMAs are free.
//   A_STEMP : the same first conv as an implicit GEMM like A_HALO, without im2col: four extra warps
//             write the 18x10 input halo patch of the tile ONCE as 32-byte pixels (16 B of bf16 hi
//             of the <= 8 channels | 16 B of bf16 lo), SWIZZLE_32B K-major layout; each tap is a
//             pair of K = 16 UMMAs on the patch shifted by (ky*10+kx) pixels (8-row group stride =
//             one patch row = 320 B), against [w_hi | w_hi] and [w_lo | 0].
//
// Warp roles (384 threads, 1 CTA / SM, persistent over tiles):
//   warp 0 : TMA producer, activations      warp 1 : MMA issuer (one elected lane)
//   warp 2 : TMEM allocator                 warp 3 : TMA producer, weights
//   warps 4-7, 8-11 : two epilogue groups (TMEM -> regs -> smem -> TMA store) taking alternate
//                     tiles, so one tile's TMEM-load / convert / store latency chain overlaps the next's
//   warps 12-19 (stem only) : two im2col producer groups
// Activations and weights have separate producers and separate mbarrier rings, so the
// activation prefetch distance (HBM latency) does not depend on the weight ring depth.
// Weight-stationary mode (`wstat`): when the whole [taps x Cin x BN] weight slab of the
// layer fits in shared memory (the Cout = 64 layers and up1), it is loaded once per CTA
// and the main loop streams activations only.
// Two to four TMEM accumulators (512 columns / BN) so the epilogue of tile i overlaps the MMAs
// of the following tiles.
//
// CTA pairs (`PAIR`, cluster of 2, tcgen05 cta_group::2): two CTAs on one TPC take two pixel
// tiles of the same column block; one UMMA of M = 256 spans both.  Each CTA stages its own
// activation patch and only HALF of the weight rows (BN/2), which halves the weight smem
// fill and cuts the shared-memory operand fetch per MMA from (128 + N) to (128 + N/2) rows
// -- the limiter of the N = 64 / 128 layers.  The leader CTA (rank 0) issues every MMA;
// "full" barriers live in the leader and count both CTAs' TMA bytes; "empty" / "accumulator
// ready" barriers are signalled in both CTAs by multicast tcgen05.commit; the peer's epilogue
// warps hand the accumulator back with remote mbarrier arrives.
#pragma once
#include "ptx.cuh"
#include "stem.cuh"

namespace ub {

enum : int { EPI_STORE = 0, EPI_STORE_POOL = 1, EPI_HEAD = 2, EPI_UPSAMPLE = 3 };
enum : int { A_TAP = 0, A_COL3 = 1, A_HALO = 2, A_STEM = 3, A_STEMP = 4, A_ROW = 5 /* conv_row.cuh */, A_PHASE = 6 /* conv_phase.cuh */, A_PS64 = 7 /* conv_ps64.cuh */ };

constexpr int kMaxClasses = 8;

// element type of the logits the head epilogues write (include/unetb200.h UNETB200_LOGITS_*): fp32 as computed, or
// the fp32 value rounded to nearest-even -- z.to(torch.float16 / torch.bfloat16) bit for bit.  The masks are always
// decided on the fp32 value.
enum : int { LOGITS_F32 = 0, LOGITS_F16 = 1, LOGITS_BF16 = 2 };

template <int LT>
__device__ __forceinline__ void store_logit(void* logits, size_t o, float z) {
    if constexpr (LT == LOGITS_F32) static_cast<float*>(logits)[o] = z;
    else if constexpr (LT == LOGITS_F16) static_cast<__half*>(logits)[o] = __float2half_rn(z);
    else static_cast<__nv_bfloat16*>(logits)[o] = __float2bfloat16_rn(z);
}
// two horizontally adjacent pixels (o even): one 8-byte (fp32) or 4-byte (16-bit) store
template <int LT>
__device__ __forceinline__ void store_logit2(void* logits, size_t o, float z0, float z1) {
    if constexpr (LT == LOGITS_F32) {
        *reinterpret_cast<float2*>(static_cast<float*>(logits) + o) = make_float2(z0, z1);
    } else if constexpr (LT == LOGITS_F16) {
        *reinterpret_cast<__half2*>(static_cast<__half*>(logits) + o) = __halves2half2(__float2half_rn(z0), __float2half_rn(z1));
    } else {
        *reinterpret_cast<__nv_bfloat162*>(static_cast<__nv_bfloat16*>(logits) + o) =
            __halves2bfloat162(__float2bfloat16_rn(z0), __float2bfloat16_rn(z1));
    }
}

// Division by a launch constant as multiply-high + shift (dividends < 2^31): the per-tile index
// arithmetic of every role (tile -> image / row / column, unit -> column block, ring slots) used ~20 %
// of the first conv's instructions as 32-bit divides.
struct FastDiv {
    uint32_t d, mul, shr;
};
inline FastDiv make_fastdiv(uint32_t d) {
    FastDiv f{d, 0u, 0u};
    if (d > 1) {
        uint32_t lg = 0;
        while ((1ull << lg) < d) ++lg;                        // ceil(log2 d)
        const uint32_t pw = 31 + lg;
        f.mul = static_cast<uint32_t>(((1ull << pw) + d - 1) / d);
        f.shr = pw - 32;
    }
    return f;
}
__device__ __forceinline__ uint32_t fdiv(uint32_t x, const FastDiv& f) {
    return f.d == 1 ? x : __umulhi(x, f.mul) >> f.shr;
}
__device__ __forceinline__ void fdivmod(uint32_t x, const FastDiv& f, int& q, int& r) {
    const uint32_t qq = fdiv(x, f);
    q = static_cast<int>(qq);
    r = static_cast<int>(x - qq * f.d);
}

struct ConvParams {
    CUtensorMap tmA0;        // source 0 activations, dims (C, W, H, N)
    CUtensorMap tmA1;        // source 1 activations (skip tensor), or == tmA0
    CUtensorMap tmB;         // weights, dims (Cin_total, rows, taps)
    CUtensorMap tmOut[4];    // output store maps ([0] for convs, [tap] for convT)
    CUtensorMap tmPool;      // pooled output store map
    CUtensorMap tmP[4];      // conv_phase.cuh: the four (row, column) parity planes of the skip tensor, dims (C, W/2, H/2, N)
    CUtensorMap tmB2;        // conv_phase.cuh: the 3x3 conv's own packed weights (skip half of K), dims (Cin_total, rows, 9)
    CUtensorMap tmB3, tmB4;  // conv_phase_stack.cuh: the 3x3 conv's weights as boxes of 64 / 32 rows x one tap (tmB / tmB2 there: the
                             // composite weights as boxes of 64 / 32 rows x one tap)
    const float* bias9;      // conv_phase.cuh: [9 border cases][Cout] fp32 (folded bias + the up-conv bias seen through the in-range taps)
    int kskip;               // conv_phase.cuh: first K column of the skip half in tmB2 (= channels of the up-conv output)
    const float* bias;       // [Cout] fp32 (BatchNorm-folded)
    const float* head_w;     // [ncls][64] fp32      (EPI_HEAD)
    const float* head_b;     // [ncls]               (EPI_HEAD)
    void* logits;            // [N][ncls][H][W], element type per the kernel's LT (EPI_HEAD, nullable)
    uint8_t* mask;           // [N][ncls][H][W] u8, or [N][ncls][H][W/8] bits when mask_bits (EPI_HEAD, nullable)
    int mask_bits;           // 1 = one bit per pixel: bit (x & 7) of byte x >> 3 of each row, LSB first
    float thr[kMaxClasses];  // logit-space thresholds
    int* dbg;                // watchdog record (nullable)
    int C0, C1;              // channels of source 0 / 1 (multiples of 64; C1 may be 0)
    int H, W, NIMG;          // spatial size of the INPUT (== output for 3x3)
    int Cout;                // output channels (per tap for convT)
    int tiles_x, tiles_y;    // ceil(W/8), ceil(H/16)
    int n_blocks;            // column blocks per pixel tile
    FastDiv fd_tpi, fd_tx, fd_nb, fd_na, fd_nout;   // dividers: tiles per image, tiles_x, n_blocks, na, n_out
    int total_tiles;
    int relu;
    int ncls;
    int na, nb;              // ring depths: activation items / weight tiles (wstat: nb = all tiles)
    int wstat;               // 1 = weight-stationary (see header)
    int n_out;               // output (and pool) staging slots PER EPILOGUE GROUP (1 or 2)
    int n_epi;               // active epilogue groups: 2 = alternate tiles, 1 = group 0 takes every tile
    int pf_items;            // activation items prefetched into L2 ahead of the smem ring (0 = off)
    int off_b, off_out, off_pool, off_bar;   // smem carve-up, bytes from the 1024-aligned base
    int off_patch;           // A_STEM: ring of TMA-loaded input halo patches + the /255 table (kStemPatchBytes)
    const void* stem_x;      // A_STEM / A_STEMP: network input (format stem_fmt), see stem.cuh
    int stem_fmt;
    const void* stem_w;      // A_STEMP: weights already in the smem tile layout (pack.cuh), 9 x 4096 B
    // conv_row.cuh: the layer's 64 bias values and the 1x1 head as KERNEL PARAMETERS, so the epilogue reads them
    // as constant-bank operands of its FADD / FFMA instead of through shared-memory loads
    float bias_c[64];
    float head_wc[kMaxClasses * 64];
    float head_bc[kMaxClasses];
};

template <int BN, int TAPS, int AMODE, bool PAIR = false>
struct ConvCfg {
    static constexpr int TPA = TAPS == 1 ? 1 : (AMODE == A_TAP ? 1 : (AMODE == A_COL3 ? 3 : 9));
    static constexpr int A_ROWS = TAPS == 1 ? 128 : (AMODE == A_TAP ? 128 : (AMODE == A_COL3 ? 144 : 180));
    static constexpr int A_TX = A_ROWS * 128;
    // A_STEMP: 180 pixels x 32 B
    static constexpr int A_STAGE = AMODE == A_STEMP ? 6144 : (A_TX + 1023) / 1024 * 1024;
    // one tap's weight rows (a CTA pair splits them); A_STEMP: two variants x 64 rows x 32 B
    static constexpr int B_TAP = AMODE == A_STEMP ? 4096 : (PAIR ? BN / 2 : BN) * 128;
    // taps per weight ring stage / per TMA box: thin per-tap tiles (<= 8 KB, A_HALO) are grouped by three so a
    // stage covers 12 MMAs and the (cross-CTA) barrier traffic drops 3x
    static constexpr int TPB = (TAPS == 9 && AMODE == A_HALO && B_TAP <= 8192) ? 3 : 1;   // (all 9 taps of a slice are one A item only in A_HALO)
    static constexpr int B_STAGE = TPB * B_TAP;
    static constexpr int NACC = BN == 256 ? 2 : 4;             // accumulator stages in TMEM
    static constexpr int TMEM_COLS = NACC * BN;                // 256 / 512 / 512 columns
};
constexpr int kStemSlots = 8;         // A_STEM: input-patch ring (TMA), slots of kStemSlotBytes
constexpr int kStemSlotBytes = 3584;  //   fp32: [Cin <= 3][18][16] floats = 3456 B; uint8: [18][48] bytes
constexpr int kStemPatchBytes = kStemSlots * kStemSlotBytes + 1024 + 2 * 2 * 3 * 180 * 4;   // ring + /255 table + split patches
// every input box of the stem (stem.cuh stem_box_bytes, Cin <= 3) fits one ring slot; fp32 NCHW is the largest
constexpr bool stem_boxes_fit(int f = 0) {
    return f == kNumXFormats ? true : (stem_box_bytes(f, 3) <= kStemSlotBytes && stem_box_bytes(f, 1) <= kStemSlotBytes &&
                                       stem_boxes_fit(f + 1));
}
static_assert(stem_boxes_fit(), "a stem input box exceeds its ring slot");
constexpr int kOutStage = 16384;      // 128 pixels x 64 channels bf16
constexpr int kPoolStage = 4096;      // 32 pixels x 64 channels bf16
constexpr int kMaxRing = 8;           // upper bound on na and (non-stationary) nb
constexpr int kBarBytes = 1024;
constexpr int kStaticSmem = 4096 + 64;   // s_bias (+ margin)
constexpr int kSmemLimit = 232448;    // 227 KB per CTA on sm_100

// X: A_STEM -> n_channels of the network input; EPI_HEAD -> n_classes (0 = generic, up to 8).
// XF: A_STEM -> input format (stem.cuh X_*; X_RUNTIME = fp32 NCHW or uint8 NHWC by p.stem_fmt).
// LT: EPI_HEAD -> logits element type (LOGITS_*).
template <int BN, int TAPS, int AMODE, int EPI, int X = 0, bool PAIR = false, int XF = X_RUNTIME, int LT = LOGITS_F32>
__global__ void __launch_bounds__(AMODE == A_STEM ? 640 : (AMODE == A_STEMP ? 512 : 384), 1)
conv_tc_kernel(const __grid_constant__ ConvParams p) {
    constexpr int CIN = X;
    static_assert(!(PAIR && (AMODE == A_STEM || AMODE == A_STEMP)), "the stem runs unpaired");
    static_assert(AMODE != A_STEMP || (TAPS == 9 && BN == 64 && CIN >= 1 && CIN <= 4 && EPI == EPI_STORE),
                  "patch stem: <= 4 input channels, 64 output channels");
    static_assert(TAPS == 9 || TAPS == 1, "3x3 conv or per-tap GEMM");
    static_assert(AMODE != A_STEM || (TAPS == 1 && BN == 64 && CIN >= 1 && 9 * CIN < 32),
                  "stem: im2col rows of < 32 taps (one K slot carries the bias), 64 output channels");
    static_assert(EPI != EPI_HEAD || BN == 64, "fused head needs all 64 channels in one tile");
    static_assert(XF == X_RUNTIME || (AMODE == A_STEM && XF != X_U8_NHWC && XF != X_F32_NCHW),
                  "compile-time input formats: the new float formats of the im2col stem");
    static_assert(LT == LOGITS_F32 || EPI == EPI_HEAD, "logits type of a head epilogue");
    using Cfg = ConvCfg<BN, TAPS, AMODE, PAIR>;
    constexpr int TPA = Cfg::TPA;
    constexpr int ITEMS = TAPS / TPA;

    extern __shared__ uint8_t smem_raw[];
    const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const uint32_t sA = smem_base;
    const uint32_t sB = smem_base + p.off_b;
    const uint32_t sOut = smem_base + p.off_out;
    const uint32_t sPool = smem_base + p.off_pool;
    const uint32_t sBar = smem_base + p.off_bar;
    const uint32_t bar_a_full = sBar;
    const uint32_t bar_a_empty = bar_a_full + 8 * kMaxRing;
    const uint32_t bar_b_full = bar_a_empty + 8 * kMaxRing;
    const uint32_t bar_b_empty = bar_b_full + 8 * kMaxRing;
    const uint32_t bar_t_full = bar_b_empty + 8 * kMaxRing;
    const uint32_t bar_t_empty = bar_t_full + 32;
    const uint32_t s_tmem_ptr = bar_t_empty + 32;
    const uint32_t bar_p_full = sBar + 512;            // A_STEM: input-patch ring
    const uint32_t bar_p_empty = bar_p_full + 8 * kStemSlots;
    uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));   // generic view of smem_base

    __shared__ __align__(16) float s_bias[1024];

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;

    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&p.tmA0);
        tma_prefetch_desc(&p.tmA1);
        tma_prefetch_desc(&p.tmB);
        if (EPI != EPI_HEAD) tma_prefetch_desc(&p.tmOut[0]);
        if (EPI == EPI_STORE_POOL) tma_prefetch_desc(&p.tmPool);
    }
    if (warp == 1 && lane == 0) {
        for (int i = 0; i < kMaxRing; ++i) {
            // full: one producer arrive per CTA of the pair (stem: every im2col thread arrives)
            mbar_init(bar_a_full + 8 * i, (AMODE == A_STEM || AMODE == A_STEMP) ? 128 : (PAIR ? 2 : 1));
            mbar_init(bar_a_empty + 8 * i, 1);
            mbar_init(bar_b_full + 8 * i, PAIR ? 2 : 1);
            mbar_init(bar_b_empty + 8 * i, 1);
        }
        for (int i = 0; i < Cfg::NACC; ++i) {
            mbar_init(bar_t_full + 8 * i, 1);
            mbar_init(bar_t_empty + 8 * i, PAIR ? 8 : 4);   // one arrive per epilogue warp (of both CTAs)
        }
        if (AMODE == A_STEM) {
            for (int i = 0; i < kStemSlots; ++i) {
                mbar_init(bar_p_full + 8 * i, 1);           // the TMA load of the patch
                mbar_init(bar_p_empty + 8 * i, 4);          // one arrive per warp of the group that read it
            }
        }
        mbar_fence_init();
    }
    if (warp == 2) {
        if (PAIR) tmem_alloc_pair<Cfg::TMEM_COLS>(s_tmem_ptr); else tmem_alloc<Cfg::TMEM_COLS>(s_tmem_ptr);
    }
    for (int i = threadIdx.x; i < p.Cout; i += blockDim.x) s_bias[i] = p.bias[i];
    tc_fence_before();
    if (PAIR) cluster_sync_all(); else __syncthreads();   // barriers of both CTAs initialised before any remote arrive
    tc_fence_after();
    const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(
        smem_gen + (s_tmem_ptr - smem_base));
    // Programmatic dependent launch: the next layer's CTAs may start as soon as SMs free up; they
    // set up, prefetch their (constant) weights and then block in pdl_wait() -- executed by the roles
    // that read the previous layer's output -- until this grid has completed.
    pdl_launch_dependents();

    const int n_cs = (p.C0 + p.C1) >> 6;            // 64-channel slices along K
    const int tiles_per_img = p.tiles_x * p.tiles_y;

    // Work units.  Unpaired: unit = (pixel tile mt, column block nb), one per CTA.  Paired: unit =
    // (pixel-tile pair, nb); CTA `rank` of the pair takes pixel tile 2*g + rank.  A pair whose second
    // tile does not exist (odd tile count) recomputes the last tile and skips its stores.
    const uint32_t rank = PAIR ? cluster_ctarank() : 0;
    const int m_tiles = tiles_per_img * p.NIMG;
    const int n_units = PAIR ? ((m_tiles + 1) >> 1) * p.n_blocks : m_tiles * p.n_blocks;
    const int first_unit = PAIR ? static_cast<int>(blockIdx.x >> 1) : static_cast<int>(blockIdx.x);
    const int unit_stride = PAIR ? static_cast<int>(gridDim.x >> 1) : static_cast<int>(gridDim.x);
    auto decode = [&](int u, int& mt, int& nb) -> bool {
        int g;
        fdivmod(static_cast<uint32_t>(u), p.fd_nb, g, nb);
        mt = PAIR ? 2 * g + static_cast<int>(rank) : g;
        const bool valid = mt < m_tiles;
        if (!valid) mt = m_tiles - 1;
        return valid;
    };

    if (AMODE == A_STEMP && warp >= 12) {
        // ============ input-patch producer (first conv, implicit GEMM) ============
        // thread r writes patch pixels q = r and q = r + 128 (< 180): 16 bytes of bf16 hi and 16
        // bytes of bf16 lo each.  No im2col: the nine taps are shifted views of this patch.
        constexpr int CI = (CIN >= 1 && CIN <= 4) ? CIN : 1;
        constexpr int D = 4;                                     // tiles of global-load prefetch (register ring)
        const int r = threadIdx.x - 384;
        const int py0 = r / 10, px0 = r % 10;                    // patch pixel q = r
        const int py1 = (r + 128) / 10, px1 = (r + 128) % 10;    // patch pixel q = r + 128 (only r < 52)
        const bool has1 = r + 128 < 180;
        auto fetch = [&](int t, float (&v)[2][CI]) {
            if (t >= p.total_tiles) return;
            int n, rr, ty_, tx_;
            fdivmod(static_cast<uint32_t>(t), p.fd_tpi, n, rr);
            fdivmod(static_cast<uint32_t>(rr), p.fd_tx, ty_, tx_);
            const int y0 = ty_ * 16 - 1, x0 = tx_ * 8 - 1;
#pragma unroll
            for (int j = 0; j < 2; ++j) {
                const int y = y0 + (j ? py1 : py0), x = x0 + (j ? px1 : px0);
                const bool in = (j == 0 || has1) && y >= 0 && y < p.H && x >= 0 && x < p.W;
#pragma unroll
                for (int ci = 0; ci < CI; ++ci) {
                    float f = 0.f;
                    if (in) {
                        if (p.stem_fmt == 0) {
                            f = __ldg(static_cast<const float*>(p.stem_x) +
                                      ((static_cast<size_t>(n) * CI + ci) * p.H + y) * p.W + x);
                        } else {
                            const uint8_t u = __ldg(static_cast<const uint8_t*>(p.stem_x) +
                                                    ((static_cast<size_t>(n) * p.H + y) * p.W + x) * CI + ci);
                            f = __fdiv_rn(static_cast<float>(u), 255.0f);   // inference.py:36 (`/ 255.0`)
                        }
                    }
                    v[j][ci] = f;
                }
            }
        };
        float ring[D][2][CI];
        pdl_wait();
        uint32_t sa = 0, pa = 0;
        const int stride = static_cast<int>(gridDim.x);
        const int t0 = static_cast<int>(blockIdx.x);
#pragma unroll
        for (int d = 0; d < D; ++d) fetch(t0 + d * stride, ring[d]);
        for (int base = t0; base < p.total_tiles; base += D * stride) {
#pragma unroll
            for (int d = 0; d < D; ++d) {
                const int t = base + d * stride;
                if (t < p.total_tiles) {
                    mbar_wait(bar_a_empty + 8 * sa, pa ^ 1, 1, p.dbg);
                    const uint32_t stage = sA + sa * Cfg::A_STAGE;
#pragma unroll
                    for (int j = 0; j < 2; ++j) {
                        if (j == 0 || has1) {
                            const int q = r + j * 128;
                            float f[4], l[4];
#pragma unroll
                            for (int ci = 0; ci < 4; ++ci) f[ci] = ci < CI ? ring[d][j][ci < CI ? ci : 0] : 0.f;
                            const uint32_t h01 = pack_bf16x2(f[0], f[1]), h23 = pack_bf16x2(f[2], f[3]);
                            l[0] = f[0] - __uint_as_float(h01 << 16);
                            l[1] = f[1] - __uint_as_float(h01 & 0xffff0000u);
                            l[2] = f[2] - __uint_as_float(h23 << 16);
                            l[3] = f[3] - __uint_as_float(h23 & 0xffff0000u);
                            // 32-byte swizzle: 16-byte chunk index ^= address bit 7 (absolute smem address)
                            const uint32_t row = stage + q * 32;
                            const uint32_t x = ((row >> 7) & 1u) << 4;
                            st_shared_v4(row + x, h01, h23, 0u, 0u);
                            st_shared_v4(row + (x ^ 16u), pack_bf16x2(l[0], l[1]), pack_bf16x2(l[2], l[3]), 0u, 0u);
                        }
                    }
                    fence_proxy_async_smem();
                    mbar_arrive(bar_a_full + 8 * sa);
                    if (++sa == static_cast<uint32_t>(p.na)) { sa = 0; pa ^= 1; }
                    fetch(t + D * stride, ring[d]);              // lands D - 1 tiles of work later
                }
            }
        }
    } else if (AMODE == A_STEM && warp >= 12) {
        // ================== im2col producer (first conv only) =================
        // thread r builds A row r = output pixel (y0 + r/8, x0 + r%8) of the tile, one ring item:
        //   k in [0,32) = bf16 hi of the 9*CIN taps (+ the constant 1.0 that meets the bias row), k in [32,64) = bf16 lo.
        // The MMA warp multiplies the whole row by [w_hi | w_hi] and the hi half again by w_lo.
        // The tile's 18 x 10 input halo patch arrives by TMA (warp 0, kStemSlots tiles ahead; out-of-image
        // elements zero-filled = the conv padding): fp32 NCHW input as [Cin][18][16] floats, uint8 NHWC input as
        // [18][48] bytes (pixel-interleaved; converted through the k / 255.0f table).  A TMA tile load FAULTS
        // (illegal instruction, measured: tools/scratch/tma_probe.cu) unless the byte offset of its innermost
        // start coordinate is a multiple of 16, so the boxes start at the 16-byte boundary below the patch's first
        // element (floats: 3 columns early; bytes: `sh` bytes early, 5 or 13 by tile parity) and are wider than
        // the 10 columns used.  Earlier versions fetched the
        // patch with per-element __ldg into registers and exchanged it through shared memory: ~95 of ~270
        // instructions per thread and tile in a kernel that is issue-bound, and the loads' latency under the
        // layer's 3 TB/s of stores showed up as the top stall of the producer warps.
        constexpr int CI = CIN > 0 ? CIN : 1;                    // (CIN == 0 only in dead instantiations)
        constexpr int KS = 9 * CI;
        constexpr int FW = 16;                                   // floats per fp32 patch row (columns 3..12 used)
        constexpr int UW = CI == 1 ? 32 : 48;                    // bytes per uint8 patch row (10 * CI used, from `sh`)
        const int grp = (threadIdx.x - 384) >> 7;                // producer group: takes tiles it % 2 == grp
        const int r = (threadIdx.x - 384) & 127;
        constexpr int PE = CI * 180;                             // patch elements: [CIN][18][10]
        constexpr int NL = (PE + 127) / 128;
        const uint8_t* s_ring = smem_gen + p.off_patch;
        float* s_lut = reinterpret_cast<float*>(smem_gen + p.off_patch + kStemSlots * kStemSlotBytes);
        // per group: two buffers of split (hi | lo) patch words
        uint32_t* s_split = reinterpret_cast<uint32_t*>(smem_gen + p.off_patch + kStemSlots * kStemSlotBytes + 1024) +
                            grp * 2 * PE;
        if (XF == X_RUNTIME && p.stem_fmt != 0) {
            // uint8 ingest: k / 255.0f (inference.py:36, IEEE division) for all 256 byte values, once per CTA
            s_lut[threadIdx.x - 384] = __fdiv_rn(static_cast<float>(threadIdx.x - 384), 255.0f);
            named_bar_sync(11, 256);
        }
        const int hh = r >> 3, ww = r & 7;
        uint32_t it = grp;                                       // CTA-local tile counter
        for (int t = static_cast<int>(blockIdx.x) + grp * static_cast<int>(gridDim.x); t < p.total_tiles;
             t += 2 * static_cast<int>(gridDim.x), it += 2) {
            const uint32_t slot = it % kStemSlots, ph = (it / kStemSlots) & 1;
            int sh = 3;                                          // first used column of the patch rows (floats)
            if (XF == X_RUNTIME ? p.stem_fmt != 0 : x_is_nhwc(XF)) {   // NHWC: (x0 - 1) * CI minus its 16-byte floor
                int n_, rr_, ty_, tx_;
                fdivmod(static_cast<uint32_t>(t), p.fd_tpi, n_, rr_);
                fdivmod(static_cast<uint32_t>(rr_), p.fd_tx, ty_, tx_);
                sh = ((tx_ * 8 - 1) * CI) & (XF == X_RUNTIME ? 15 : x_per_16B(XF) - 1);
            }
            mbar_wait(bar_p_full + 8 * slot, ph, 2, p.dbg);
            const uint8_t* pb = s_ring + slot * kStemSlotBytes + (p.stem_fmt != 0 ? sh : 0);
            const float* pf = reinterpret_cast<const float*>(s_ring + slot * kStemSlotBytes) + 3;
            // pass 1: every patch element is converted and split into bf16 hi | lo ONCE (not once per tap that
            // uses it: 540 splits per tile instead of 3 456) and parked as one packed word, [ci][18][10]
            uint32_t* p2 = s_split + (it & 2 ? PE : 0);          // (it advances by 2: alternate buffers)
#pragma unroll
            for (int i = 0; i < NL; ++i) {
                const int e = r + i * 128;
                if (e < PE) {
                    const int ci = e / 180, rem = e - ci * 180, py = rem / 10, px = rem - py * 10;
                    float v;
                    if constexpr (XF == X_RUNTIME) {
                        v = p.stem_fmt == 0 ? pf[(ci * 18 + py) * FW + px] : s_lut[pb[py * UW + px * CI + ci]];
                    } else {
                        // the element in its format (box geometry: stem.cuh stem_box_w), widened to fp32 -- exact, so
                        // from here on the same bits as the fp32 NCHW path on x.float()
                        constexpr int BW = stem_box_w(XF, CI);
                        const int i = x_is_nhwc(XF) ? py * BW + sh + px * CI + ci
                                                    : (ci * 18 + py) * BW + (x_per_16B(XF) - 1) + px;
                        const uint8_t* box = s_ring + slot * kStemSlotBytes;
                        if constexpr (x_elem_bytes(XF) == 4) v = reinterpret_cast<const float*>(box)[i];
                        else v = x_widen16<XF>(reinterpret_cast<const uint16_t*>(box)[i]);
                    }
                    const uint32_t h2 = pack_bf16x2(v, 0.f);                           // hi in the low half
                    const uint32_t l2 = pack_bf16x2(v - __uint_as_float(h2 << 16), 0.f);
                    p2[e] = __byte_perm(h2, l2, 0x5410);                                // hi | lo << 16
                }
            }
            named_bar_sync(9 + grp, 128);
            if (lane == 0) mbar_arrive(bar_p_empty + 8 * slot);  // (after the barrier: every warp is done with the patch)
            // pass 2: this pixel's K row: 27 packed words -> hi pairs and lo pairs by byte permutes
            uint32_t hi[16], lo[16];                             // 32 bf16 each, zero padded past KS + 1
#pragma unroll
            for (int k2 = 0; k2 < 16; ++k2) {
                uint32_t w2[2];
#pragma unroll
                for (int j = 0; j < 2; ++j) {
                    const int k = 2 * k2 + j;
                    if (k < KS) {
                        const int tap = k / CI, ci = k - tap * CI;
                        w2[j] = p2[ci * 180 + (hh + tap / 3) * 10 + (ww + tap % 3)];
                    } else {
                        // first pad slot = constant 1.0 (hi = 0x3F80, lo = 0): its weight row holds the folded bias
                        // (pack.cuh), so the GEMM adds it and the stem's (issue-bound) epilogue does not
                        w2[j] = k == KS ? 0x00003F80u : 0u;
                    }
                }
                hi[k2] = __byte_perm(w2[0], w2[1], 0x5410);
                lo[k2] = __byte_perm(w2[0], w2[1], 0x7632);
            }
            // ring item of this CTA-local tile
            {
                const uint32_t qa = fdiv(it, p.fd_na);
                const uint32_t sa = it - qa * p.fd_na.d, pa = qa & 1;
                mbar_wait(bar_a_empty + 8 * sa, pa ^ 1, 1, p.dbg);
                const uint32_t row = sA + sa * Cfg::A_STAGE + r * 128;
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    st_shared_v4(row + ((c ^ (r & 7)) << 4), hi[4 * c], hi[4 * c + 1], hi[4 * c + 2], hi[4 * c + 3]);
                    st_shared_v4(row + (((c + 4) ^ (r & 7)) << 4), lo[4 * c], lo[4 * c + 1], lo[4 * c + 2], lo[4 * c + 3]);
                }
                fence_proxy_async_smem();
                mbar_arrive(bar_a_full + 8 * sa);
            }
        }
    } else if (warp == 0 && AMODE == A_STEM) {
        // ============ TMA producer: input halo patches of the first conv ============
        if (lane == 0) {
            constexpr int CI = CIN > 0 ? CIN : 1;
            constexpr uint32_t kBytes32 = CI * 18 * 16 * 4, kBytes8 = 18 * (CI == 1 ? 32 : 48);
            pdl_wait();
            uint32_t it = 0;
            for (int t = static_cast<int>(blockIdx.x); t < p.total_tiles; t += static_cast<int>(gridDim.x), ++it) {
                const uint32_t slot = it % kStemSlots, ph = (it / kStemSlots) & 1;
                int n, rr, ty_, tx_;
                fdivmod(static_cast<uint32_t>(t), p.fd_tpi, n, rr);
                fdivmod(static_cast<uint32_t>(rr), p.fd_tx, ty_, tx_);
                const int y0 = ty_ * 16 - 1, x0 = tx_ * 8 - 1;
                mbar_wait(bar_p_empty + 8 * slot, ph ^ 1, 1, p.dbg);
                const uint32_t dst = smem_base + p.off_patch + slot * kStemSlotBytes;
                // (the innermost start coordinate must sit on a 16-byte boundary, see the im2col producer)
                if constexpr (XF != X_RUNTIME) {                 // box geometry: stem.cuh stem_box_w
                    mbar_expect_tx(bar_p_full + 8 * slot, stem_box_bytes(XF, CI));
                    if (x_is_nhwc(XF))
                        tma_load_3d(dst, &p.tmA0, bar_p_full + 8 * slot, (x0 * CI) & ~(x_per_16B(XF) - 1), y0, n);
                    else
                        tma_load_4d(dst, &p.tmA0, bar_p_full + 8 * slot, x0 - (x_per_16B(XF) - 1), y0, 0, n);
                } else if (p.stem_fmt == 0) {                           // fp32 [N][C][H][W]: box 16 x 18 x Cin from x0 - 3
                    mbar_expect_tx(bar_p_full + 8 * slot, kBytes32);
                    tma_load_4d(dst, &p.tmA0, bar_p_full + 8 * slot, x0 - 3, y0, 0, n);
                } else {                                         // uint8 [N][H][W * Cin]: box 48 (32) bytes x 18
                    mbar_expect_tx(bar_p_full + 8 * slot, kBytes8);
                    tma_load_3d(dst, &p.tmA0, bar_p_full + 8 * slot, (x0 * CI) & ~15, y0, n);
                }
            }
        }
    } else if (warp == 0) {
        // ===================== TMA producer: activations ======================
        if (lane == 0 && AMODE != A_STEM && AMODE != A_STEMP) {
            // flat walk over this CTA's activation items: idx -> (tile, 64-channel slice, item)
            const int ipt = n_cs * ITEMS;
            const int my_units = first_unit < n_units ? (n_units - first_unit + unit_stride - 1) / unit_stride : 0;
            const int n_items = my_units * ipt;
            auto locate = [&](int idx, const CUtensorMap*& tm, int& ca, int& bx, int& by, int& n) {
                const int tl = idx / ipt, rem = idx - tl * ipt;
                const int cs = rem / ITEMS, item = rem - cs * ITEMS;
                int mt, nb_unused;
                decode(first_unit + tl * unit_stride, mt, nb_unused);
                int r;
                fdivmod(static_cast<uint32_t>(mt), p.fd_tpi, n, r);
                fdivmod(static_cast<uint32_t>(r), p.fd_tx, by, bx);
                by *= 16;
                bx *= 8;
                const bool src0 = (cs << 6) < p.C0;
                tm = src0 ? &p.tmA0 : &p.tmA1;
                ca = src0 ? (cs << 6) : (cs << 6) - p.C0;
                if (TAPS == 9) {
                    if (AMODE == A_TAP) { bx += item % 3 - 1; by += item / 3 - 1; }
                    if (AMODE == A_COL3) { bx += item - 1; by -= 1; }
                    if (AMODE == A_HALO) { bx -= 1; by -= 1; }
                }
            };
            const CUtensorMap* tm;
            int ca, bx, by, n;
            pdl_wait();
            const int pf = p.pf_items;
            for (int i = 0; i < pf && i < n_items; ++i) {
                locate(i, tm, ca, bx, by, n);
                tma_prefetch_4d(tm, ca, bx, by, n);
            }
            uint32_t sa = 0, pa = 0;
            for (int i = 0; i < n_items; ++i) {
                if (pf > 0 && i + pf < n_items) {
                    locate(i + pf, tm, ca, bx, by, n);
                    tma_prefetch_4d(tm, ca, bx, by, n);
                }
                locate(i, tm, ca, bx, by, n);
                mbar_wait(bar_a_empty + 8 * sa, pa ^ 1, 1, p.dbg);
                if (PAIR) {
                    // both CTAs' bytes are counted on the leader's barrier
                    const uint32_t fb = mapa_shared(bar_a_full + 8 * sa, 0);
                    if (rank == 0) mbar_expect_tx(bar_a_full + 8 * sa, 2 * Cfg::A_TX); else mbar_arrive_cluster(fb);
                    tma_load_4d_pair(sA + sa * Cfg::A_STAGE, tm, fb, ca, bx, by, n);
                } else {
                    mbar_expect_tx(bar_a_full + 8 * sa, Cfg::A_TX);
                    tma_load_4d(sA + sa * Cfg::A_STAGE, tm, bar_a_full + 8 * sa, ca, bx, by, n);
                }
                if (++sa == static_cast<uint32_t>(p.na)) { sa = 0; pa ^= 1; }
            }
        }
    } else if (warp == 3) {
        // ======================= TMA producer: weights ========================
        if (AMODE == A_STEMP) {
            // 36 KB of first-conv weights, already in the smem tile layout: plain copy by the warp
            const uint4* src = static_cast<const uint4*>(p.stem_w);
            for (int i = lane; i < 9 * Cfg::B_TAP / 16; i += 32) {
                const uint4 w4 = __ldg(src + i);
                st_shared_v4(sB + i * 16, w4.x, w4.y, w4.z, w4.w);
            }
            fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) mbar_arrive(bar_b_full);
        } else if (lane == 0) {
            const int row_off = PAIR ? static_cast<int>(rank) * (BN / 2) : 0;   // this CTA's half of the weight rows
            if (p.wstat) {
                // whole weight slab of this layer, once: slot = cs * TAPS + tap
                // (stem: two K slices of weights, [w_hi | w_hi] and [w_lo | 0], for its single activation slice)
                const int n_wcs = AMODE == A_STEM ? 2 : n_cs;
                const uint32_t bytes = static_cast<uint32_t>(n_wcs * TAPS) * Cfg::B_TAP;
                const uint32_t fb = PAIR ? mapa_shared(bar_b_full, 0) : bar_b_full;
                if (!PAIR) mbar_expect_tx(bar_b_full, bytes);
                else if (rank == 0) mbar_expect_tx(bar_b_full, 2 * bytes);
                else mbar_arrive_cluster(fb);
                for (int cs = 0; cs < n_wcs; ++cs)
                    for (int tap = 0; tap < TAPS; tap += Cfg::TPB) {      // one box = TPB consecutive taps
                        const uint32_t dst = sB + (cs * TAPS + tap) * Cfg::B_TAP;
                        if (PAIR) tma_load_3d_pair(dst, &p.tmB, fb, cs << 6, row_off, tap);
                        else tma_load_3d(dst, &p.tmB, fb, cs << 6, 0, tap);
                    }
            } else {
                uint32_t sb = 0, pb = 0;
                for (int u = first_unit; u < n_units; u += unit_stride) {
                    const int nb = u - static_cast<int>(fdiv(static_cast<uint32_t>(u), p.fd_nb)) * p.n_blocks;
                    for (int cs = 0; cs < n_cs; ++cs) {
#pragma unroll 1
                        for (int i = 0; i < TAPS; i += Cfg::TPB) {
                            // same tap order as the MMA loop (A_COL3 walks column-major, TPB == 1 there)
                            const int tap = (TAPS == 9 && AMODE == A_COL3) ? (i % 3) * 3 + i / 3 : i;
                            mbar_wait(bar_b_empty + 8 * sb, pb ^ 1, 3, p.dbg);
                            if (PAIR) {
                                const uint32_t fb = mapa_shared(bar_b_full + 8 * sb, 0);
                                if (rank == 0) mbar_expect_tx(bar_b_full + 8 * sb, 2 * Cfg::B_STAGE);
                                else mbar_arrive_cluster(fb);
                                tma_load_3d_pair(sB + sb * Cfg::B_STAGE, &p.tmB, fb, cs << 6,
                                                 nb * BN + row_off, tap);
                            } else {
                                mbar_expect_tx(bar_b_full + 8 * sb, Cfg::B_STAGE);
                                tma_load_3d(sB + sb * Cfg::B_STAGE, &p.tmB, bar_b_full + 8 * sb, cs << 6,
                                            nb * BN, tap);
                            }
                            if (++sb == static_cast<uint32_t>(p.nb)) { sb = 0; pb ^= 1; }
                        }
                    }
                }
            }
        }
    } else if (warp == 1) {
        // ============================ MMA issuer ==============================
        // One lane issues every tcgen05.mma of the CTA.  For N <= 128 an MMA retires in
        // 32-64 cycles, so the issue path itself is kept to a couple of integer ops per MMA:
        // descriptor high words are constants, low words are (base + constant) in 16-byte
        // units, and mbarrier probes for the next stage are issued ahead of the MMAs.
        // The whole warp walks the loops converged (uniform addresses live in uniform registers);
        // one elected lane issues the MMAs and commits.
        if (AMODE == A_STEMP) {
            // patch stem: per tile 9 taps x {[w_hi | w_hi], [w_lo | 0]} K = 16 UMMAs on shifted patch views.
            // SWIZZLE_32B K-major descriptors: rows (pixels / output channels) are 32 B, the 8-row
            // group stride is one patch row (320 B) for A and 256 B for B.
            constexpr uint32_t idesc = umma_idesc_bf16(BN, 128);
            constexpr uint32_t a_hi = umma_desc_hi_sw32(320), b_hi = umma_desc_hi_sw32(256);
            uint32_t sa = 0, pa = 0, tile_it = 0;
            mbar_wait(bar_b_full, 0, 8, p.dbg);
            tc_fence_after();
            const uint32_t b_lo0 = umma_desc_lo(sB);
            for (int u = first_unit; u < n_units; u += unit_stride, ++tile_it) {
                const uint32_t acc = tile_it % Cfg::NACC, acc_ph = (tile_it / Cfg::NACC) & 1;
                mbar_wait(bar_t_empty + 8 * acc, acc_ph ^ 1, 4, p.dbg);
                mbar_wait(bar_a_full + 8 * sa, pa, 5, p.dbg);
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + acc * BN;
                const uint32_t a_lo0 = umma_desc_lo(sA + sa * Cfg::A_STAGE);
                if (elect_one()) {
#pragma unroll
                    for (int tap = 0; tap < 9; ++tap) {
                        const uint32_t a_lo = a_lo0 + 2 * ((tap / 3) * 10 + (tap % 3));   // one pixel = two 16-byte units
#pragma unroll
                        for (int v = 0; v < 2; ++v)
                            umma_bf16(d_tmem, umma_desc(a_lo, a_hi),
                                      umma_desc(b_lo0 + (tap * 2 + v) * (2048 >> 4), b_hi), idesc, (tap | v) ? 1u : 0u);
                    }
                    umma_commit(bar_a_empty + 8 * sa);
                    umma_commit(bar_t_full + 8 * acc);
                }
                if (++sa == static_cast<uint32_t>(p.na)) { sa = 0; pa ^= 1; }
            }
        } else if (rank == 0) {
            constexpr uint32_t idesc = umma_idesc_bf16(BN, PAIR ? 256 : 128);
            constexpr uint32_t a_sbo = (TAPS == 9 && AMODE == A_HALO) ? 10 * 128 : 1024;
            constexpr uint32_t a_hi = umma_desc_hi_sw128(a_sbo);
            constexpr uint32_t b_hi = umma_desc_hi_sw128(1024);
            uint32_t sa = 0, pa = 0, sb = 0, pb = 0, tile_it = 0;
            if (p.wstat) {
                mbar_wait(bar_b_full, 0, 8, p.dbg);
                tc_fence_after();
            }
            const uint32_t b_lo0 = umma_desc_lo(sB);
            for (int u = first_unit; u < n_units; u += unit_stride, ++tile_it) {
                const uint32_t acc = tile_it % Cfg::NACC, acc_ph = (tile_it / Cfg::NACC) & 1;
                mbar_wait(bar_t_empty + 8 * acc, acc_ph ^ 1, 4, p.dbg);
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + acc * BN;
                uint32_t accumulate = 0;
                for (int cs = 0; cs < n_cs; ++cs) {
#pragma unroll 1
                    for (int item = 0; item < ITEMS; ++item) {
                        mbar_wait(bar_a_full + 8 * sa, pa, 5, p.dbg);
                        tc_fence_after();
                        const uint32_t a_lo0 = umma_desc_lo(sA + sa * Cfg::A_STAGE);
                        const bool last_item = (cs == n_cs - 1) && (item == ITEMS - 1);
                        auto mma = [&](uint32_t a_lo, uint32_t b_lo, uint32_t acc_flag) {
                            if (PAIR) umma_bf16_pair(d_tmem, umma_desc(a_lo, a_hi), umma_desc(b_lo, b_hi), idesc, acc_flag);
                            else umma_bf16(d_tmem, umma_desc(a_lo, a_hi), umma_desc(b_lo, b_hi), idesc, acc_flag);
                        };
                        auto commit = [&](uint32_t bar) {
                            if (PAIR) umma_commit_pair(bar); else umma_commit(bar);
                        };
                        // activation view of tap tt inside the staged item, in 16-byte units
                        auto a_view = [&](int tt) -> uint32_t {
                            return TAPS == 1 ? 0u
                                 : (AMODE == A_COL3 ? static_cast<uint32_t>(tt) * (1024 >> 4)
                                 : (AMODE == A_HALO ? static_cast<uint32_t>((tt / 3) * 10 + (tt % 3)) * (128 >> 4) : 0u));
                        };
                        if (p.wstat) {
                            // resident weights (slot = cs * TAPS + tap): every MMA of the item back to back
                            const uint32_t b_cs = b_lo0 + (cs * TAPS) * (Cfg::B_TAP >> 4);
                            if (elect_one()) {
#pragma unroll
                                for (int tt = 0; tt < TPA; ++tt) {
                                    const int tap_c = TAPS == 1 ? 0 : (AMODE == A_COL3 ? tt * 3 : tt);
                                    const uint32_t tap_r = (TAPS == 9 && AMODE != A_HALO) ? item * (AMODE == A_COL3 ? 1 : TPA) : 0;
                                    const uint32_t b_lo = b_cs + (tap_c + tap_r) * (Cfg::B_TAP >> 4);
#pragma unroll
                                    for (int k = 0; k < 4; ++k)
                                        mma(a_lo0 + a_view(tt) + 2 * k, b_lo + 2 * k, (tt | k) ? 1u : accumulate);
                                }
                                if (AMODE == A_STEM) {
                                    // x_hi * w_lo: the hi half of the row (K = 32) against the second weight slice
#pragma unroll
                                    for (int k = 0; k < 2; ++k)
                                        mma(a_lo0 + 2 * k, b_lo0 + (Cfg::B_TAP >> 4) + 2 * k, 1u);
                                }
                                commit(bar_a_empty + 8 * sa);
                                if (last_item) commit(bar_t_full + 8 * acc);
                            }
                            accumulate = 1;
                        } else {
                            constexpr int TPB = Cfg::TPB;
                            bool ready = mbar_try_wait(bar_b_full + 8 * sb, pb);
#pragma unroll
                            for (int st = 0; st < TPA / TPB; ++st) {
                                if (!ready) mbar_wait(bar_b_full + 8 * sb, pb, 6, p.dbg);
                                tc_fence_after();
                                const uint32_t b_stage_lo = b_lo0 + sb * (Cfg::B_STAGE >> 4);
                                const uint32_t cur = sb;
                                if (++sb == static_cast<uint32_t>(p.nb)) { sb = 0; pb ^= 1; }
                                // probe the next weight stage now; the answer is needed after these MMAs
                                ready = mbar_try_wait(bar_b_full + 8 * sb, pb);
                                if (elect_one()) {
#pragma unroll
                                    for (int j = 0; j < TPB; ++j) {
                                        const int tt = st * TPB + j;
#pragma unroll
                                        for (int k = 0; k < 4; ++k)
                                            mma(a_lo0 + a_view(tt) + 2 * k, b_stage_lo + j * (Cfg::B_TAP >> 4) + 2 * k,
                                                (j | k) ? 1u : accumulate);
                                    }
                                    commit(bar_b_empty + 8 * cur);
                                    if (st == TPA / TPB - 1) {
                                        commit(bar_a_empty + 8 * sa);
                                        if (last_item) commit(bar_t_full + 8 * acc);
                                    }
                                }
                                accumulate = 1;
                            }
                        }
                        if (++sa == static_cast<uint32_t>(p.na)) { sa = 0; pa ^= 1; }
                    }
                }
            }
        }
    } else if (warp >= 4 && warp < 12) {
        // ============================= epilogue ===============================
        const int eg = (warp - 4) >> 2;         // epilogue group: takes tiles tile_it % 2 == eg
        const int q = warp & 3;                 // TMEM lane quarter this warp may access (warp id % 4)
        const int row = q * 32 + lane;          // pixel row of the tile: h = row/8, w = row%8
        const int estep = p.n_epi;              // tiles between two tiles of this group
        // BN == 64 launches (one 64-column chunk per tile, in production a single column block): the
        // chunk's 64 bias values live in registers and are reloaded only when the channel offset
        // changes (the thin-K epilogues stalled on their shared-memory loads)
        constexpr bool kBiasRegs = BN == 64 && AMODE != A_STEM && AMODE != A_STEMP && EPI != EPI_HEAD;   // (the 640-thread stem has 102 registers per thread; the head reads its bias as kernel parameters)
        float bias_r[kBiasRegs ? 64 : 1];
        int bias_ch0 = -1;
        auto load_bias = [&](int ch0) {
            if (kBiasRegs && ch0 != bias_ch0) {
#pragma unroll
                for (int i = 0; i < (kBiasRegs ? 64 : 1); ++i) bias_r[i] = s_bias[ch0 + i];
                bias_ch0 = ch0;
            }
        };
        uint32_t tile_it = eg, chunk_it = 0;
        // hand-back of an accumulator: arrive on the (leader's) barrier the MMA issuer waits on
        auto release_acc = [&](uint32_t acc) {
            if (PAIR) mbar_arrive_cluster(mapa_shared(bar_t_empty + 8 * acc, 0));
            else mbar_arrive(bar_t_empty + 8 * acc);
        };
        for (int u = eg < estep ? first_unit + eg * unit_stride : n_units; u < n_units;
             u += estep * unit_stride, tile_it += estep) {
            int mt, nb;
            const bool valid = decode(u, mt, nb);
            int n, r, y0, x0;
            fdivmod(static_cast<uint32_t>(mt), p.fd_tpi, n, r);
            fdivmod(static_cast<uint32_t>(r), p.fd_tx, y0, x0);
            y0 *= 16;
            x0 *= 8;
            const uint32_t acc = tile_it % Cfg::NACC, acc_ph = (tile_it / Cfg::NACC) & 1;
            mbar_wait(bar_t_full + 8 * acc, acc_ph, 7, p.dbg);
            tc_fence_after();
            const uint32_t t_addr = tmem_base + acc * BN + (static_cast<uint32_t>(q * 32) << 16);

            if (EPI == EPI_HEAD) {
                // out_conv 1x1 (unet_model.py:86) from the fp32 accumulators, NC classes at once.  Bias and head
                // weights are kernel parameters (ConvParams::bias_c / head_wc / head_bc, zero past n_classes): every
                // use below is a constant-bank operand -- no registers, no shared-memory loads in the FFMA stream
                constexpr int NC = X > 0 ? X : kMaxClasses;
                float z[NC];
#pragma unroll
                for (int c = 0; c < NC; ++c) z[c] = p.head_bc[c];
#pragma unroll
                for (int half = 0; half < 2; ++half) {
                    uint32_t v[32];
                    tmem_ld32(t_addr + half * 32, v);
                    tmem_ld_wait();
#pragma unroll
                    for (int i = 0; i < 32; i += 4) {
                        float f0 = __uint_as_float(v[i + 0]) + p.bias_c[half * 32 + i];
                        float f1 = __uint_as_float(v[i + 1]) + p.bias_c[half * 32 + i + 1];
                        float f2 = __uint_as_float(v[i + 2]) + p.bias_c[half * 32 + i + 2];
                        float f3 = __uint_as_float(v[i + 3]) + p.bias_c[half * 32 + i + 3];
                        if (p.relu) {
                            f0 = fmaxf(f0, 0.f);
                            f1 = fmaxf(f1, 0.f);
                            f2 = fmaxf(f2, 0.f);
                            f3 = fmaxf(f3, 0.f);
                        }
#pragma unroll
                        for (int c = 0; c < NC; ++c) {
                            const int k0 = c * 64 + half * 32 + i;
                            z[c] = fmaf(f0, p.head_wc[k0], z[c]);
                            z[c] = fmaf(f1, p.head_wc[k0 + 1], z[c]);
                            z[c] = fmaf(f2, p.head_wc[k0 + 2], z[c]);
                            z[c] = fmaf(f3, p.head_wc[k0 + 3], z[c]);
                        }
                    }
                }
                tc_fence_before();
                __syncwarp();
                if (lane == 0) release_acc(acc);
                const int y = y0 + (row >> 3), x = x0 + (row & 7);
                const bool inside = valid && y < p.H && x < p.W;
                if (inside) {
#pragma unroll
                    for (int c = 0; c < NC; ++c) {
                        if (c < p.ncls) {
                            const size_t o = ((static_cast<size_t>(n) * p.ncls + c) * p.H + y) * p.W + x;
                            if (p.logits) store_logit<LT>(p.logits, o, z[c]);
                            if (p.mask && !p.mask_bits) p.mask[o] = z[c] > p.thr[c] ? 1 : 0;
                        }
                    }
                }
                if (p.mask && p.mask_bits) {
                    // one bit per pixel (inference.py:75-79 keeps a boolean per pixel): the warp's 32 pixels are
                    // 4 tile rows x 8 columns, x0 is a multiple of 8 and W of 16, so byte r of the ballot is
                    // exactly byte x0 / 8 of image row y0 + 4q + r.  Lanes 0..3 store one byte each.
#pragma unroll
                    for (int c = 0; c < NC; ++c) {
                        const uint32_t bits = __ballot_sync(0xffffffffu, inside && z[c] > p.thr[c]);
                        const int yr = y0 + 4 * q + lane;
                        if (c < p.ncls && lane < 4 && valid && yr < p.H && x0 < p.W)
                            p.mask[((static_cast<size_t>(n) * p.ncls + c) * p.H + yr) * (p.W >> 3) + (x0 >> 3)] =
                                static_cast<uint8_t>(bits >> (8 * lane));
                    }
                }
            }

#pragma unroll 1
            for (int j = 0; j < (EPI == EPI_HEAD ? 0 : BN / 64); ++j, ++chunk_it) {
                const int gcol = nb * BN + j * 64;            // global column of this 64-wide chunk
                const int tapo = EPI == EPI_UPSAMPLE ? gcol / p.Cout : 0;
                const int ch0 = EPI == EPI_UPSAMPLE ? gcol - tapo * p.Cout : gcol;
                load_bias(ch0);
                // Each warp owns a quarter of the tile (4 pixel rows): its own 4 KB slab of the staging
                // slot, its own TMA stores, its own bulk groups -- no barrier between the four warps.
                // Each group owns n_out slots; a slab was last read by this warp's store n_out chunks ago.
                const uint32_t buf = eg * p.n_out + (chunk_it - fdiv(chunk_it, p.fd_nout) * p.fd_nout.d);
                const uint32_t obuf = sOut + buf * kOutStage;
                const uint32_t pbuf = sPool + buf * kPoolStage;
                if (lane == 0) {
                    if (p.n_out == 2) tma_store_wait_read<1>(); else tma_store_wait_read<0>();
                }
                __syncwarp();
                uint32_t pk[32];
#pragma unroll
                for (int half = 0; half < 2; ++half) {
                    uint32_t v[32];
                    tmem_ld32(t_addr + j * 64 + half * 32, v);
                    tmem_ld_wait();
#pragma unroll
                    for (int i = 0; i < 32; i += 4) {
                        float4 b4;
                        if (AMODE == A_STEM) {
                            b4 = make_float4(0.f, 0.f, 0.f, 0.f);    // bias already added by the GEMM (constant-one K slot)
                        } else if (kBiasRegs) {
                            constexpr int o = kBiasRegs ? 1 : 0;     // (keeps the indices in range otherwise)
                            b4 = make_float4(bias_r[o * (half * 32 + i)], bias_r[o * (half * 32 + i + 1)],
                                             bias_r[o * (half * 32 + i + 2)], bias_r[o * (half * 32 + i + 3)]);
                        } else {
                            b4 = *reinterpret_cast<const float4*>(s_bias + ch0 + half * 32 + i);
                        }
                        float f0 = __uint_as_float(v[i + 0]) + b4.x;
                        float f1 = __uint_as_float(v[i + 1]) + b4.y;
                        float f2 = __uint_as_float(v[i + 2]) + b4.z;
                        float f3 = __uint_as_float(v[i + 3]) + b4.w;
                        if (p.relu) {
                            f0 = fmaxf(f0, 0.f);
                            f1 = fmaxf(f1, 0.f);
                            f2 = fmaxf(f2, 0.f);
                            f3 = fmaxf(f3, 0.f);
                        }
                        pk[half * 16 + i / 2] = pack_bf16x2(f0, f1);
                        pk[half * 16 + i / 2 + 1] = pack_bf16x2(f2, f3);
                    }
                }
                if (j == BN / 64 - 1) {   // accumulator fully drained -> hand it back to the MMA warp
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) release_acc(acc);
                }
#pragma unroll
                for (int c16 = 0; c16 < 8; ++c16)
                    st_shared_v4(obuf + row * 128 + ((c16 ^ (row & 7)) << 4), pk[c16 * 4],
                                 pk[c16 * 4 + 1], pk[c16 * 4 + 2], pk[c16 * 4 + 3]);
                if (EPI == EPI_STORE_POOL) {
                    // 2x2 max-pool: partners are lane^1 (x) and lane^8 (y); bf16 rounding is
                    // monotone, so max of rounded == rounded max (unet_model.py:34,57).
#pragma unroll
                    for (int i = 0; i < 32; ++i) {
                        uint32_t m = max_bf16x2(pk[i], __shfl_xor_sync(0xffffffffu, pk[i], 1));
                        pk[i] = max_bf16x2(m, __shfl_xor_sync(0xffffffffu, m, 8));
                    }
                    if ((lane & 9) == 0) {
                        const int pr = (q * 2 + (lane >> 4)) * 4 + ((lane & 7) >> 1);
#pragma unroll
                        for (int c16 = 0; c16 < 8; ++c16)
                            st_shared_v4(pbuf + pr * 128 + ((c16 ^ (pr & 7)) << 4), pk[c16 * 4],
                                         pk[c16 * 4 + 1], pk[c16 * 4 + 2], pk[c16 * 4 + 3]);
                    }
                }
                fence_proxy_async_smem();
                __syncwarp();
                if (lane == 0) {
                    if (valid) {
                        // this warp's rows y0 + 4q .. +3 (pooled: (y0 >> 1) + 2q, +1)
                        if (EPI == EPI_UPSAMPLE)
                            tma_store_4d(&p.tmOut[tapo], obuf + q * 4096, ch0, x0, y0 + 4 * q, n);
                        else
                            tma_store_4d(&p.tmOut[0], obuf + q * 4096, ch0, x0, y0 + 4 * q, n);
                        if (EPI == EPI_STORE_POOL)
                            tma_store_4d(&p.tmPool, pbuf + q * 1024, ch0, x0 >> 1, (y0 >> 1) + 2 * q, n);
                    }
                    tma_store_commit();
                }
            }
        }
        if (lane == 0) tma_store_wait_all<0>();
    }

    tc_fence_before();
    if (PAIR) cluster_sync_all(); else __syncthreads();   // the peer may still signal this CTA's barriers until here
    if (warp == 2) {
        tc_fence_after();
        if (PAIR) tmem_dealloc_pair<Cfg::TMEM_COLS>(tmem_base); else tmem_dealloc<Cfg::TMEM_COLS>(tmem_base);
    }
}

}  // namespace ub
