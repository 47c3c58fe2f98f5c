// 3x3 convolution with 64 output channels as a ROW-STACKED implicit GEMM (tcgen05 + TMEM + TMA).
//
// Why a second kernel.  conv_tc_kernel issues nine UMMAs of N = Cout per 64-channel K slice, one per tap, each
// re-reading the 128 x 16 activation operand from shared memory.  For Cout = 64 that operand fetch alone is
// 4 KB per 32-cycle UMMA = the whole 128 B/clk of shared-memory bandwidth, so down1.net.3, conv1.net.0 and
// conv1.net.3 (unet_model.py:29,48 -- 20 % of the network's FLOPs) sat at 69-74 % tensor-pipe activity against a
// ceiling of 80 % (profiles/r01d_ncu_summary_table.md).  The only way past it is more output columns per
// activation fetch, and a 64-channel layer has no more channels -- but it has more TAPS:
//
//   GEMM rows (M = 128)  = 128 consecutive pixels of ONE image row (x), so the three kx taps are row shifts of
//                          the staged input row (start address + kx * 128 B, canonical SWIZZLE_128B layout);
//   GEMM columns (N)     = the three ky taps stacked: B = [W(ky=2,kx); W(ky=1,kx); W(ky=0,kx)], 192 rows;
//   accumulators (TMEM)  = R = 4 output rows side by side, 64 columns each.  Input row i of the tile's
//                          (R + 2)-row halo contributes to output rows i-2, i-1, i through ky = 2, 1, 0 -- which
//                          are ADJACENT accumulator column groups -- so one UMMA of N = 192 at column offset
//                          64 * (i - 2) adds all three.  The first / last rows of the halo use the N = 64 / 128
//                          sub-ranges of the same weight block.
//
// One activation fetch now feeds N = 192 columns: 10 KB of operands per 96-cycle UMMA (107 B/clk) instead of
// 5 KB per 32 cycles, and the MMA count per tile drops 2.4x.  Per output element the K order is unchanged
// (slice -> ky -> kx -> 16-channel step), so results are bit-identical to conv_tc_kernel's.
// An accumulator group's first touch must overwrite (UMMA accumulate = 0) while the other groups of the same
// UMMA accumulate, so the first UMMA of halo rows 0..3 is split in two (N = 64 with accumulate 0 + the rest).
//
// Unpaired (cta_group::1): a CTA pair splits B by N halves, which would interleave the ky groups of the two
// CTAs in the accumulator columns; with N = 192 the B fetch no longer limits anyway.
//
// Warp roles (384 threads, 1 CTA / SM, persistent over tiles of 4 rows x 128 pixels):
//   warp 0 : TMA producer, one item per (K slice, halo row): box 64 ch x 130 pixels (zero fill = padding)
//   warp 1 : MMA issuer          warp 2 : TMEM allocator (2 accumulators x 4 rows x 64 columns; handing the rows
//            over one by one -- row barriers instead of tile barriers -- was measured 10 % SLOWER)
//   warp 3 : weights, once: the whole [slice][kx][ky = 2,1,0][64][64] slab stays resident
//   warps 4-7, 8-11 : two epilogue groups, each draining half of the rows of EVERY tile; a warp owns 32 pixels
//                     of its rows.
#pragma once
#include "conv_tc.cuh"

namespace ub {

constexpr int kRowR = 4;                               // output rows per tile
constexpr int kRowW = 128;                             // output pixels per tile row = UMMA M
constexpr int kRowItemBytes = (kRowW + 2) * 128;       // one halo row of one K slice
constexpr int kRowAStage = (kRowItemBytes + 1023) / 1024 * 1024;
constexpr int kRowBBlock = 64 * 128;                   // one tap of one K slice: 64 couts x 64 cin bf16
constexpr int kRowStatic = 64;                         // static shared memory of the kernel (none; margin)

template <int EPI, int X = 0, int LT = LOGITS_F32>   // LT: logits element type of EPI_HEAD (conv_tc.cuh)
__global__ void __launch_bounds__(384, 1) conv_row_kernel(const __grid_constant__ ConvParams p) {
    static_assert(EPI == EPI_STORE || EPI == EPI_STORE_POOL || EPI == EPI_HEAD, "row kernel epilogues");
    constexpr int R = kRowR;
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
    const uint32_t bar_t_full = bar_b_full + 8;
    const uint32_t bar_t_empty = bar_t_full + 16;
    const uint32_t s_tmem_ptr = bar_t_empty + 16;
    uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));

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
            mbar_init(bar_a_full + 8 * i, 1);
            mbar_init(bar_a_empty + 8 * i, 1);
        }
        mbar_init(bar_b_full, 1);
        for (int i = 0; i < 2; ++i) {
            mbar_init(bar_t_full + 8 * i, 1);
            mbar_init(bar_t_empty + 8 * i, 4 * p.n_epi);   // one arrive per active epilogue warp
        }
        mbar_fence_init();
    }
    if (warp == 2) tmem_alloc<512>(s_tmem_ptr);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(smem_gen + (s_tmem_ptr - smem_base));
    pdl_launch_dependents();          // see conv_tc.cuh: the next layer may set up while this one runs

    const int n_cs = (p.C0 + p.C1) >> 6;
    const int first_tile = static_cast<int>(blockIdx.x), tile_stride = static_cast<int>(gridDim.x);
    auto decode = [&](int t, int& n, int& y0, int& x0) {
        int r;
        fdivmod(static_cast<uint32_t>(t), p.fd_tpi, n, r);
        fdivmod(static_cast<uint32_t>(r), p.fd_tx, y0, x0);
        y0 *= R;
        x0 *= kRowW;
    };

    if (warp == 0) {
        // ===================== TMA producer: halo rows of the activations ======================
        if (lane == 0) {
            pdl_wait();
            uint32_t sa = 0, pa = 0;
            for (int t = first_tile; t < p.total_tiles; t += tile_stride) {
                int n, y0, x0;
                decode(t, n, y0, x0);
                for (int cs = 0; cs < n_cs; ++cs) {
                    const bool src0 = (cs << 6) < p.C0;
                    const CUtensorMap* tm = src0 ? &p.tmA0 : &p.tmA1;
                    const int ca = src0 ? (cs << 6) : (cs << 6) - p.C0;
                    for (int i = 0; i < R + 2; ++i) {
                        mbar_wait(bar_a_empty + 8 * sa, pa ^ 1, 1, p.dbg);
                        mbar_expect_tx(bar_a_full + 8 * sa, kRowItemBytes);
                        tma_load_4d(sA + sa * kRowAStage, tm, bar_a_full + 8 * sa, ca, x0 - 1, y0 - 1 + i, n);
                        if (++sa == static_cast<uint32_t>(p.na)) { sa = 0; pa ^= 1; }
                    }
                }
            }
        }
    } else if (warp == 3) {
        // ======================= weights: resident slab, loaded once ========================
        // smem block ((cs * 3 + kx) * 3 + g) holds tap (ky = 2 - g, kx) of K slice cs, so the three ky taps of
        // one kx are 192 consecutive B rows in the order the accumulator column groups need
        if (lane == 0) {
            mbar_expect_tx(bar_b_full, static_cast<uint32_t>(n_cs * 9) * kRowBBlock);
            for (int cs = 0; cs < n_cs; ++cs)
                for (int kx = 0; kx < 3; ++kx)
                    for (int ky = 0; ky < 3; ++ky)
                        tma_load_3d(sB + ((cs * 3 + kx) * 3 + (2 - ky)) * kRowBBlock, &p.tmB, bar_b_full, cs << 6, 0,
                                    ky * 3 + kx);
        }
    } else if (warp == 1) {
        // ============================ MMA issuer ==============================
        constexpr uint32_t d_hi = umma_desc_hi_sw128(1024);
        constexpr uint32_t kBlk = kRowBBlock >> 4;                 // one weight block in 16-byte units
        uint32_t sa = 0, pa = 0, tile_it = 0;
        mbar_wait(bar_b_full, 0, 8, p.dbg);
        tc_fence_after();
        const uint32_t b_lo0 = umma_desc_lo(sB);
        for (int t = first_tile; t < p.total_tiles; t += tile_stride, ++tile_it) {
            const uint32_t acc = tile_it & 1, acc_ph = (tile_it >> 1) & 1;
            mbar_wait(bar_t_empty + 8 * acc, acc_ph ^ 1, 4, p.dbg);
            tc_fence_after();
            const uint32_t d0 = tmem_base + acc * (R * 64);
            for (int cs = 0; cs < n_cs; ++cs) {
                const uint32_t b_cs = b_lo0 + static_cast<uint32_t>(cs * 9) * kBlk;
                const bool last_cs = cs == n_cs - 1;
#pragma unroll
                for (int i = 0; i < R + 2; ++i) {
                    // halo row i feeds output rows i - ky, ky in [ky_min, ky_max]; B blocks g = 2 - ky
                    constexpr int dummy = 0;
                    (void)dummy;
                    const int ky_max = i < 2 ? i : 2;
                    const int ky_min = i - (R - 1) > 0 ? i - (R - 1) : 0;
                    const int ng = ky_max - ky_min + 1;                       // accumulator groups touched
                    const uint32_t g0 = static_cast<uint32_t>(2 - ky_max);    // first weight block
                    const uint32_t dcol = d0 + 64u * static_cast<uint32_t>(i - ky_max);
                    mbar_wait(bar_a_full + 8 * sa, pa, 5, p.dbg);
                    tc_fence_after();
                    const uint32_t a_lo0 = umma_desc_lo(sA + sa * kRowAStage);
                    if (elect_one()) {
#pragma unroll
                        for (int kx = 0; kx < 3; ++kx) {
#pragma unroll
                            for (int k = 0; k < 4; ++k) {
                                const uint64_t ad = umma_desc(a_lo0 + kx * (128 >> 4) + 2 * k, d_hi);
                                const uint32_t b_lo = b_cs + static_cast<uint32_t>(kx * 3) * kBlk + 2 * k;
                                if (kx == 0 && k == 0 && i < R && cs == 0) {
                                    // first touch of output row i (its ky = 0 group): overwrite it, accumulate the rest
                                    if (ng > 1)
                                        umma_bf16(dcol, ad, umma_desc(b_lo + g0 * kBlk, d_hi),
                                                  umma_idesc_bf16(64 * (ng - 1), 128), 1u);
                                    umma_bf16(dcol + 64u * (ng - 1), ad, umma_desc(b_lo + 2 * kBlk, d_hi),
                                              umma_idesc_bf16(64, 128), 0u);
                                } else {
                                    umma_bf16(dcol, ad, umma_desc(b_lo + g0 * kBlk, d_hi), umma_idesc_bf16(64 * ng, 128), 1u);
                                }
                            }
                        }
                        umma_commit(bar_a_empty + 8 * sa);
                        if (last_cs && i == R + 1) umma_commit(bar_t_full + 8 * acc);
                    }
                    if (++sa == static_cast<uint32_t>(p.na)) { sa = 0; pa ^= 1; }
                }
            }
        }
    } else if (warp >= 4) {
        // ============================= epilogue ===============================
        // Both epilogue groups work on EVERY tile, half of its rows each (group 0: rows 0-1, group 1: rows 2-3):
        // with only two accumulators in TMEM the UMMAs of tile t + 2 wait for tile t to be drained, so what
        // counts is the drain LATENCY of one tile, not the throughput of two tiles drained side by side
        // (alternate tiles per group, the conv_tc.cuh scheme, left the MMA warp waiting ~20 % of the time).
        const int eg = (warp - 4) >> 2;         // epilogue group
        const int q = warp & 3;                 // TMEM lane quarter = pixels 32q .. 32q + 31 of the tile row
        const int j_lo = p.n_epi == 2 ? eg * (R / 2) : 0;
        const int j_hi = p.n_epi == 2 ? j_lo + R / 2 : R;
        uint32_t tile_it = 0, chunk_it = 0;
        // bias and head weights are kernel parameters (ConvParams::bias_c / head_wc): with the loops below fully
        // unrolled every use is a constant-bank operand, no registers and no shared-memory loads
        for (int t = eg < p.n_epi ? first_tile : p.total_tiles; t < p.total_tiles; t += tile_stride, ++tile_it) {
            int n, y0, x0;
            decode(t, n, y0, x0);
            const uint32_t acc = tile_it & 1, acc_ph = (tile_it >> 1) & 1;
            mbar_wait(bar_t_full + 8 * acc, acc_ph, 7, p.dbg);
            tc_fence_after();
            const uint32_t t_addr = tmem_base + acc * (R * 64) + (static_cast<uint32_t>(q * 32) << 16);
            auto row_ready = [&](int) {};            // (accumulators are handed over per tile, see the header)
            auto row_done = [&](int j) {             // this warp's last row read: its share of the accumulator is free
                if (j == j_hi - 1) {
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(bar_t_empty + 8 * acc);
                }
            };
            const int xw = x0 + 32 * q;          // first pixel of this warp
            const int px = xw + lane;            // this thread's pixel

            if (EPI == EPI_HEAD) {
                constexpr int NC = X > 0 ? X : kMaxClasses;
#pragma unroll 1
                for (int j = j_lo; j < j_hi; ++j) {
                    row_ready(j);
                    float z[NC];
#pragma unroll
                    for (int c = 0; c < NC; ++c) z[c] = p.head_bc[c];
#pragma unroll
                    for (int half = 0; half < 2; ++half) {
                        uint32_t v[32];
                        tmem_ld32(t_addr + j * 64 + half * 32, v);
                        tmem_ld_wait();
                        if (half == 1) row_done(j);
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
                    const int y = y0 + j;
                    const bool inside = y < p.H && px < p.W;
                    if (inside) {
#pragma unroll
                        for (int c = 0; c < NC; ++c) {
                            if (c < p.ncls) {
                                const size_t o = ((static_cast<size_t>(n) * p.ncls + c) * p.H + y) * p.W + px;
                                if (p.logits) store_logit<LT>(p.logits, o, z[c]);
                                if (p.mask && !p.mask_bits) p.mask[o] = z[c] > p.thr[c] ? 1 : 0;
                            }
                        }
                    }
                    if (p.mask && p.mask_bits) {
                        // 32 consecutive pixels of one row = 4 bytes of the bit plane; lanes 0..3 store one each
#pragma unroll
                        for (int c = 0; c < NC; ++c) {
                            const uint32_t bits = __ballot_sync(0xffffffffu, inside && z[c] > p.thr[c]);
                            if (c < p.ncls && lane < 4 && y < p.H && xw + 8 * lane < p.W)
                                p.mask[((static_cast<size_t>(n) * p.ncls + c) * p.H + y) * (p.W >> 3) + (xw >> 3) + lane] =
                                    static_cast<uint8_t>(bits >> (8 * lane));
                        }
                    }
                }
            } else if (EPI == EPI_STORE) {
#pragma unroll 1
                for (int j = j_lo; j < j_hi; ++j, ++chunk_it) {
                    // a warp owns its 32 pixels of the row: its own 4 KB slab of the slot, its own TMA stores
                    const uint32_t slot = chunk_it - fdiv(chunk_it, p.fd_nout) * p.fd_nout.d;
                    const uint32_t slab = sOut + (eg * p.n_out + slot) * kOutStage + q * 4096;
                    if (lane == 0) {
                        if (p.n_out == 2) tma_store_wait_read<1>(); else tma_store_wait_read<0>();
                    }
                    __syncwarp();
                    row_ready(j);
                    uint32_t pk[32];
#pragma unroll
                    for (int half = 0; half < 2; ++half) {
                        uint32_t v[32];
                        tmem_ld32(t_addr + j * 64 + half * 32, v);
                        tmem_ld_wait();
                        if (half == 1) row_done(j);
#pragma unroll
                        for (int i = 0; i < 32; i += 2) {
                            float f0 = __uint_as_float(v[i + 0]) + p.bias_c[half * 32 + i];
                            float f1 = __uint_as_float(v[i + 1]) + p.bias_c[half * 32 + i + 1];
                            if (p.relu) {
                                f0 = fmaxf(f0, 0.f);
                                f1 = fmaxf(f1, 0.f);
                            }
                            pk[half * 16 + i / 2] = pack_bf16x2(f0, f1);
                        }
                    }
#pragma unroll
                    for (int c16 = 0; c16 < 8; ++c16)
                        st_shared_v4(slab + lane * 128 + ((c16 ^ (lane & 7)) << 4), pk[c16 * 4], pk[c16 * 4 + 1],
                                     pk[c16 * 4 + 2], pk[c16 * 4 + 3]);
                    fence_proxy_async_smem();
                    __syncwarp();
                    if (lane == 0) {
                        if (y0 + j < p.H && xw < p.W) tma_store_4d(&p.tmOut[0], slab, 0, xw, y0 + j, n);
                        tma_store_commit();
                    }
                }
            } else {
                // EPI_STORE_POOL: rows 2jp and 2jp + 1 together, so the 2x2 max-pool (unet_model.py:34,57) is a
                // register max of the two rows + one shuffle with the x neighbour; bf16 rounding is monotone, so
                // max of rounded == rounded max.  Slots 0 / 1 of the group take the two rows.
#pragma unroll 1
                for (int jp = j_lo / 2; jp < j_hi / 2; ++jp) {
                    const uint32_t slab_a = sOut + (eg * 2 + 0) * kOutStage + q * 4096;
                    const uint32_t slab_b = sOut + (eg * 2 + 1) * kOutStage + q * 4096;
                    const uint32_t pslab = sPool + eg * 8192 + q * 2048;
                    if (lane == 0) tma_store_wait_read<0>();
                    __syncwarp();
                    row_ready(2 * jp);
                    row_ready(2 * jp + 1);
#pragma unroll
                    for (int half = 0; half < 2; ++half) {
                        uint32_t va[32], vb[32], pa_[16], pb_[16];
                        tmem_ld32(t_addr + (2 * jp) * 64 + half * 32, va);
                        tmem_ld32(t_addr + (2 * jp + 1) * 64 + half * 32, vb);
                        tmem_ld_wait();
                        if (half == 1) {
                            row_done(2 * jp);
                            row_done(2 * jp + 1);
                        }
#pragma unroll
                        for (int i = 0; i < 32; i += 4) {
                            const float4 b4 = make_float4(p.bias_c[half * 32 + i], p.bias_c[half * 32 + i + 1],
                                                          p.bias_c[half * 32 + i + 2], p.bias_c[half * 32 + i + 3]);
                            float a0 = __uint_as_float(va[i + 0]) + b4.x, a1 = __uint_as_float(va[i + 1]) + b4.y;
                            float a2 = __uint_as_float(va[i + 2]) + b4.z, a3 = __uint_as_float(va[i + 3]) + b4.w;
                            float c0 = __uint_as_float(vb[i + 0]) + b4.x, c1 = __uint_as_float(vb[i + 1]) + b4.y;
                            float c2 = __uint_as_float(vb[i + 2]) + b4.z, c3 = __uint_as_float(vb[i + 3]) + b4.w;
                            if (p.relu) {
                                a0 = fmaxf(a0, 0.f); a1 = fmaxf(a1, 0.f); a2 = fmaxf(a2, 0.f); a3 = fmaxf(a3, 0.f);
                                c0 = fmaxf(c0, 0.f); c1 = fmaxf(c1, 0.f); c2 = fmaxf(c2, 0.f); c3 = fmaxf(c3, 0.f);
                            }
                            pa_[i / 2] = pack_bf16x2(a0, a1);
                            pa_[i / 2 + 1] = pack_bf16x2(a2, a3);
                            pb_[i / 2] = pack_bf16x2(c0, c1);
                            pb_[i / 2 + 1] = pack_bf16x2(c2, c3);
                        }
#pragma unroll
                        for (int cc = 0; cc < 4; ++cc) {
                            const int c16 = half * 4 + cc;
                            st_shared_v4(slab_a + lane * 128 + ((c16 ^ (lane & 7)) << 4), pa_[cc * 4], pa_[cc * 4 + 1],
                                         pa_[cc * 4 + 2], pa_[cc * 4 + 3]);
                            st_shared_v4(slab_b + lane * 128 + ((c16 ^ (lane & 7)) << 4), pb_[cc * 4], pb_[cc * 4 + 1],
                                         pb_[cc * 4 + 2], pb_[cc * 4 + 3]);
                        }
#pragma unroll
                        for (int i = 0; i < 16; ++i) {
                            const uint32_t m = max_bf16x2(pa_[i], pb_[i]);
                            pa_[i] = max_bf16x2(m, __shfl_xor_sync(0xffffffffu, m, 1));
                        }
                        if ((lane & 1) == 0) {
                            const int pr = lane >> 1;
#pragma unroll
                            for (int cc = 0; cc < 4; ++cc) {
                                const int c16 = half * 4 + cc;
                                st_shared_v4(pslab + pr * 128 + ((c16 ^ (pr & 7)) << 4), pa_[cc * 4], pa_[cc * 4 + 1],
                                             pa_[cc * 4 + 2], pa_[cc * 4 + 3]);
                            }
                        }
                    }
                    fence_proxy_async_smem();
                    __syncwarp();
                    if (lane == 0) {
                        const int y = y0 + 2 * jp;
                        if (xw < p.W) {
                            if (y < p.H) tma_store_4d(&p.tmOut[0], slab_a, 0, xw, y, n);
                            if (y + 1 < p.H) tma_store_4d(&p.tmOut[0], slab_b, 0, xw, y + 1, n);
                            if (y + 1 < p.H) tma_store_4d(&p.tmPool, pslab, 0, xw >> 1, y >> 1, n);
                        }
                        tma_store_commit();
                    }
                }
            }
        }
        if (lane == 0) tma_store_wait_all<0>();
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 2) {
        tc_fence_after();
        tmem_dealloc<512>(tmem_base);
    }
}

}  // namespace ub
