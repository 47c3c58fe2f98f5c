// 3x3 convolution 64 -> 64 channels as a PHASE-STACKED implicit GEMM (tcgen05 + TMEM + TMA, CTA pairs).
//
// Why.  A UMMA of N = 64 reads 4 KB of activations and 1 KB of weights from shared memory for 32 cycles of tensor
// work: 160 B/clk against the ~128 B/clk the SM delivers, so down1.net.3 and conv1.net.3 (unet_model.py:29,48) sit
// at 72 % tensor-pipe activity in conv_tc_kernel whatever else is tuned (DESIGN.md, "Where the 64-channel layers
// stand").  The only way out is more output columns per activation fetch, and a 64-channel layer has no more
// channels -- but neighbouring output PIXELS read the same input pixel through different taps:
//
//   split the output into its four parities (py, px) of 2x2 blocks ("phases", as in conv_phase.cuh) and the input
//   into its four parity planes (qy, qx).  Output (2I + py, 2J + px) reads, through tap (ky, kx), input pixel
//   (2I + r, 2J + c) with r = py + ky - 1, c = px + kx - 1 in {-1, 0, 1, 2}: position (I + (r >> 1), J + (c >> 1)) of
//   plane (r & 1, c & 1).  So ONE shifted view (r, c) of a staged plane box is the A operand of up to FOUR
//   (phase, tap) products: both py when r is 0 or 1, both px when c is 0 or 1.
//
// GEMM rows (M = 128 per CTA, 256 per pair) = 16 x 8 block positions (I, J) = a 32 x 16 pixel tile; the four phases
// are four 64-column groups of one 256-column accumulator (ph = 2 py + px), so phases (py, 0), (py, 1) are ADJACENT
// and one UMMA of N = 128 feeds both from one activation fetch.  Per 16-channel K step and view:
//   r, c in {0,1}   : 2 UMMAs of N = 128   [(ph0,ph1) <- taps (r+1, c+1 | c);  (ph2,ph3) <- taps (r, c+1 | c)]
//   r in {0,1}, c = -1 | 2 : 2 UMMAs of N = 64 (phases px = 0 | 1 of both py: not adjacent)
//   r = -1 | 2, c in {0,1} : 1 UMMA of N = 128 (py = 0 | 1)         corners : 1 UMMA of N = 64
// = 24 activation fetches instead of 36 per K step and 512 output pixels, 132 KB instead of 180 KB of operands.
//
// Weights stay resident.  In a CTA pair each CTA supplies HALF of a UMMA's B rows from ITS OWN shared memory at the
// descriptor's address, so the two CTAs hold different images: for the N = 128 UMMAs CTA 0 supplies the px = 0
// phase (tap kx = c + 1) and CTA 1 the px = 1 phase (tap kx = c) -- image 1, slot (ky, j): tap (ky, j + 1) in CTA 0,
// tap (ky, j) in CTA 1, all 64 rows; for the N = 64 UMMAs both supply 32 rows of the same tap -- image 2, slot
// (ky, kx / 2) for kx in {0, 2}.  72 KB per CTA.
//
// Per output element the K order differs from conv_tc_kernel's (taps are visited plane by plane), so results agree
// to fp32 accumulation-order noise, not bit for bit.
//
// Warp roles as in conv_tc.cuh: warp 0 = TMA producer (one plane box, 18 x 10 positions, per ring slot), warp 1 = MMA
// issuer (static schedule: one elect block of 24 UMMAs per plane), warp 2 = TMEM allocator, warp 3 = weights (once),
// warps 4-11 = epilogue groups.  Epilogues: EPI_STORE_POOL (four phase stores through strided maps + the 2x2 max-pool,
// which is a thread-local max over the four phases) and EPI_HEAD (out_conv + threshold on the fp32 accumulators).
#pragma once
#include "conv_tc.cuh"

namespace ub {

constexpr int kPsBoxW = 10, kPsBoxH = 18;
constexpr int kPsBoxTx = kPsBoxW * kPsBoxH * 128;                 // one plane box: 23 040 B
constexpr int kPsSlot = (kPsBoxTx + 1023) / 1024 * 1024;
constexpr int kPsW1 = 6 * 8192;                                   // image 1: six whole taps (64 rows x 128 B)
constexpr int kPsW2 = 6 * 4096;                                   // image 2: six half taps (32 rows)
constexpr int kPsWBytes = kPsW1 + kPsW2;
constexpr int kPsStatic = 64;

template <int EPI, int X = 0, int LT = LOGITS_F32>   // LT: logits element type of EPI_HEAD (conv_tc.cuh)
__global__ void __launch_bounds__(384, 1) conv_ps64_kernel(const __grid_constant__ ConvParams p) {
    static_assert(EPI == EPI_STORE || EPI == EPI_STORE_POOL || EPI == EPI_HEAD, "phase-stacked kernel epilogues");
    extern __shared__ uint8_t smem_raw[];
    const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const uint32_t sA = smem_base;
    const uint32_t sB = smem_base + p.off_b;
    const uint32_t sOut = smem_base + p.off_out;
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
    const uint32_t rank = cluster_ctarank();

    if (warp == 0 && lane == 0) {
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            tma_prefetch_desc(&p.tmP[q]);
            if (EPI != EPI_HEAD) tma_prefetch_desc(&p.tmOut[q]);
        }
        tma_prefetch_desc(&p.tmB);
        tma_prefetch_desc(&p.tmB2);
        if (EPI == EPI_STORE_POOL) tma_prefetch_desc(&p.tmPool);
    }
    if (warp == 1 && lane == 0) {
        for (int i = 0; i < kMaxRing; ++i) {
            mbar_init(bar_a_full + 8 * i, 2);
            mbar_init(bar_a_empty + 8 * i, 1);
        }
        mbar_init(bar_b_full, 2);
        for (int i = 0; i < 2; ++i) {
            mbar_init(bar_t_full + 8 * i, 1);
            mbar_init(bar_t_empty + 8 * i, 8);       // one arrive per epilogue warp of the group, in both CTAs
        }
        mbar_fence_init();
    }
    if (warp == 2) tmem_alloc_pair<512>(s_tmem_ptr);
    tc_fence_before();
    cluster_sync_all();
    tc_fence_after();
    const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(smem_gen + (s_tmem_ptr - smem_base));
    pdl_launch_dependents();

    // work unit = a pair of 16 x 8 block-position tiles (CTA `rank` takes tile 2 g + rank); an odd tail recomputes
    // the last tile and skips its stores
    const int m_tiles = p.tiles_x * p.tiles_y * p.NIMG;
    const int n_units = (m_tiles + 1) >> 1;
    const int first_unit = static_cast<int>(blockIdx.x >> 1), unit_stride = static_cast<int>(gridDim.x >> 1);
    auto decode = [&](int u, int& n, int& y0, int& x0) -> bool {
        int mt = 2 * u + static_cast<int>(rank);
        const bool valid = mt < m_tiles;
        if (!valid) mt = m_tiles - 1;
        int r;
        fdivmod(static_cast<uint32_t>(mt), p.fd_tpi, n, r);
        fdivmod(static_cast<uint32_t>(r), p.fd_tx, y0, x0);
        y0 *= 16;
        x0 *= 8;
        return valid;
    };

    if (warp == 0) {
        // ===================== TMA producer: the four parity planes of the input, one box per slot ======================
        if (lane == 0) {
            pdl_wait();
            uint32_t sa = 0, pa = 0;
            for (int u = first_unit; u < n_units; u += unit_stride) {
                int n, y0, x0;
                decode(u, n, y0, x0);
#pragma unroll 1
                for (int q = 0; q < 4; ++q) {
                    mbar_wait(bar_a_empty + 8 * sa, pa ^ 1, 1, p.dbg);
                    const uint32_t fb = mapa_shared(bar_a_full + 8 * sa, 0);
                    if (rank == 0) mbar_expect_tx(bar_a_full + 8 * sa, 2 * kPsBoxTx); else mbar_arrive_cluster(fb);
                    tma_load_4d_pair(sA + sa * kPsSlot, &p.tmP[q], fb, 0, x0 - 1, y0 - 1, n);
                    if (++sa == static_cast<uint32_t>(p.na)) { sa = 0; pa ^= 1; }
                }
            }
        }
    } else if (warp == 3) {
        // ======================= weights: the two resident images of this CTA, loaded once ========================
        if (lane == 0) {
            const uint32_t fb = mapa_shared(bar_b_full, 0);
            if (rank == 0) mbar_expect_tx(bar_b_full, 2 * kPsWBytes); else mbar_arrive_cluster(fb);
            for (int ky = 0; ky < 3; ++ky)
                for (int j = 0; j < 2; ++j) {
                    // image 1, slot (ky, j): whole tap (ky, j + 1) in CTA 0, (ky, j) in CTA 1
                    tma_load_3d_pair(sB + (ky * 2 + j) * 8192, &p.tmB, fb, 0, 0, ky * 3 + j + (rank == 0 ? 1 : 0));
                    // image 2, slot (ky, j): rows 32 rank .. + 31 of tap (ky, 2 j)
                    tma_load_3d_pair(sB + kPsW1 + (ky * 2 + j) * 4096, &p.tmB2, fb, 0, static_cast<int>(rank) * 32,
                                     ky * 3 + 2 * j);
                }
        }
    } else if (warp == 1) {
        // ============================ MMA issuer (leader CTA) ==============================
        if (rank == 0) {
            constexpr uint32_t idesc128 = umma_idesc_bf16(128, 256), idesc64 = umma_idesc_bf16(64, 256);
            constexpr uint32_t a_hi = umma_desc_hi_sw128(kPsBoxW * 128);
            constexpr uint32_t b_hi = umma_desc_hi_sw128(1024);
            uint32_t sa = 0, pa = 0, tile_it = 0;
            mbar_wait(bar_b_full, 0, 8, p.dbg);
            tc_fence_after();
            const uint32_t b1 = umma_desc_lo(sB), b2 = umma_desc_lo(sB + kPsW1);
            for (int u = first_unit; u < n_units; u += unit_stride, ++tile_it) {
                const uint32_t acc = tile_it & 1, acc_ph = (tile_it >> 1) & 1;
                mbar_wait(bar_t_empty + 8 * acc, acc_ph ^ 1, 4, p.dbg);
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + acc * 256;
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const int qy = q >> 1, qx = q & 1;
                    mbar_wait(bar_a_full + 8 * sa, pa, 5, p.dbg);
                    tc_fence_after();
                    const uint32_t a0 = umma_desc_lo(sA + sa * kPsSlot);
                    if (elect_one()) {
#pragma unroll
                        for (int iy = 0; iy < 2; ++iy)
#pragma unroll
                            for (int ix = 0; ix < 2; ++ix) {
                                const int r = 2 * iy - qy, c = 2 * ix - qx;        // qy = 0: r = 0, 2;  qy = 1: r = -1, 1
                                const uint32_t av = a0 + static_cast<uint32_t>(((r >> 1) + 1) * kPsBoxW + ((c >> 1) + 1)) * 8;
                                const bool fresh = q == 0 && iy == 0 && ix == 0;   // view (0, 0) touches every phase first
                                const bool rmid = r == 0 || r == 1, cmid = c == 0 || c == 1;
                                // N = 128 over phases (py, 0), (py, 1): image-1 slot (ky, c)
                                auto mma128 = [&](int py, int ky) {
#pragma unroll
                                    for (int k = 0; k < 4; ++k)
                                        umma_bf16_pair(d_tmem + py * 128, umma_desc(av + 2 * k, a_hi),
                                                       umma_desc(b1 + (ky * 2 + c) * (8192 >> 4) + 2 * k, b_hi), idesc128,
                                                       (fresh && k == 0) ? 0u : 1u);
                                };
                                // N = 64 over phase (py, px): image-2 slot (ky, px)   [kx = 2 px: c = -1 -> px 0, c = 2 -> px 1]
                                auto mma64 = [&](int py, int px, int ky) {
#pragma unroll
                                    for (int k = 0; k < 4; ++k)
                                        umma_bf16_pair(d_tmem + (py * 2 + px) * 64, umma_desc(av + 2 * k, a_hi),
                                                       umma_desc(b2 + (ky * 2 + px) * (4096 >> 4) + 2 * k, b_hi), idesc64, 1u);
                                };
                                if (cmid) {
                                    if (rmid) { mma128(0, r + 1); mma128(1, r); }
                                    else if (r < 0) mma128(0, 0);
                                    else mma128(1, 2);
                                } else {
                                    const int px = c < 0 ? 0 : 1;
                                    if (rmid) { mma64(0, px, r + 1); mma64(1, px, r); }
                                    else if (r < 0) mma64(0, px, 0);
                                    else mma64(1, px, 2);
                                }
                            }
                        umma_commit_pair(bar_a_empty + 8 * sa);
                        if (q == 3) umma_commit_pair(bar_t_full + 8 * acc);
                    }
                    if (++sa == static_cast<uint32_t>(p.na)) { sa = 0; pa ^= 1; }
                }
            }
        }
    } else if (warp >= 4) {
        // ============================= epilogue ===============================
        const int eg = (warp - 4) >> 2;         // epilogue group: takes units tile_it % n_epi == eg
        const int q = warp & 3;                 // TMEM lane quarter
        const int row = q * 32 + lane;          // block position of the tile: I = y0 + row / 8, J = x0 + row % 8
        const int estep = p.n_epi;
        uint32_t tile_it = eg, chunk_it = 0;
        auto release_acc = [&](uint32_t acc) { mbar_arrive_cluster(mapa_shared(bar_t_empty + 8 * acc, 0)); };
        for (int u = eg < estep ? first_unit + eg * unit_stride : n_units; u < n_units;
             u += estep * unit_stride, tile_it += estep) {
            int n, y0, x0;
            const bool valid = decode(u, n, y0, x0);
            const uint32_t acc = tile_it & 1, acc_ph = (tile_it >> 1) & 1;
            mbar_wait(bar_t_full + 8 * acc, acc_ph, 7, p.dbg);
            tc_fence_after();
            const uint32_t t_addr = tmem_base + acc * 256 + (static_cast<uint32_t>(q * 32) << 16);
            const int I = y0 + (row >> 3), J = x0 + (row & 7);

            if (EPI == EPI_HEAD) {
                // out_conv 1x1 (unet_model.py:86) from the fp32 accumulators; bias / head weights are kernel parameters
                constexpr int NC = X > 0 ? X : kMaxClasses;
                const int HW2 = p.W >> 1;                         // block positions per image row
                const bool inside = valid && I < (p.H >> 1) && J < HW2;
                // one wait per phase (64 columns by a tcgen05.ld pair) instead of one per 32 columns: the epilogue is
                // latency-bound, and with two waits per phase the MMA warp waited for accumulators (ncu: 25 spins per unit)
                uint32_t v[64];
                auto load_phase = [&](int ph) {
                    tmem_ld32(t_addr + ph * 64, *reinterpret_cast<uint32_t(*)[32]>(&v[0]));
                    tmem_ld32(t_addr + ph * 64 + 32, *reinterpret_cast<uint32_t(*)[32]>(&v[32]));
                };
                load_phase(0);
#pragma unroll 1
                for (int py = 0; py < 2; ++py) {
                    float z[2][NC];
#pragma unroll
                    for (int px = 0; px < 2; ++px) {
#pragma unroll
                        for (int c = 0; c < NC; ++c) z[px][c] = p.head_bc[c];
                        tmem_ld_wait();
#pragma unroll
                        for (int i = 0; i < 64; ++i) {
                            float f = __uint_as_float(v[i]) + p.bias_c[i];
                            if (p.relu) f = fmaxf(f, 0.f);
#pragma unroll
                            for (int c = 0; c < NC; ++c) z[px][c] = fmaf(f, p.head_wc[c * 64 + i], z[px][c]);
                        }
                        if (py * 2 + px < 3) load_phase(py * 2 + px + 1);     // in flight while this phase's outputs are written
                    }
                    if (py == 1) {                                // accumulator fully read -> hand it back
                        tc_fence_before();
                        __syncwarp();
                        if (lane == 0) release_acc(acc);
                    }
                    const int y = 2 * I + py, x = 2 * J;
#pragma unroll
                    for (int c = 0; c < NC; ++c) {
                        if (c < p.ncls && inside) {
                            const size_t o = ((static_cast<size_t>(n) * p.ncls + c) * p.H + y) * p.W + x;
                            if (p.logits) store_logit2<LT>(p.logits, o, z[0][c], z[1][c]);
                            if (p.mask && !p.mask_bits)
                                *reinterpret_cast<uchar2*>(p.mask + o) =
                                    make_uchar2(z[0][c] > p.thr[c] ? 1 : 0, z[1][c] > p.thr[c] ? 1 : 0);
                        }
                    }
                    if (p.mask && p.mask_bits) {
                        // one bit per pixel: the warp's 32 positions are 4 block rows x 8 block columns = 16 pixels of
                        // image rows 2 (y0 + 4 q + i) + py; bit 2 j + px of those 16 = position j of ballot px.
                        // Lanes 0..3 interleave one row each and store its two bytes (x0 is a multiple of 8 positions).
#pragma unroll
                        for (int c = 0; c < NC; ++c) {
                            const uint32_t b0 = __ballot_sync(0xffffffffu, inside && z[0][c] > p.thr[c]);
                            const uint32_t b1 = __ballot_sync(0xffffffffu, inside && z[1][c] > p.thr[c]);
                            const int Ir = y0 + 4 * q + lane;
                            if (c < p.ncls && lane < 4 && valid && Ir < (p.H >> 1) && x0 < HW2) {
                                uint32_t e = (b0 >> (8 * lane)) & 0xffu, o = (b1 >> (8 * lane)) & 0xffu, w = 0;
#pragma unroll
                                for (int j = 0; j < 8; ++j) w |= (((e >> j) & 1u) << (2 * j)) | (((o >> j) & 1u) << (2 * j + 1));
                                *reinterpret_cast<uint16_t*>(p.mask + ((static_cast<size_t>(n) * p.ncls + c) * p.H + 2 * Ir + py) *
                                                                          (p.W >> 3) + (x0 >> 2)) = static_cast<uint16_t>(w);
                            }
                        }
                    }
                }
            } else {
                // four phase tiles (+ the pooled tile): TMEM -> bias / ReLU -> bf16 -> swizzled staging -> TMA store.
                // p.n_out staging slots per group in rotation (3 with one group, 2 with two): a slot was last read by
                // the store n_out chunks ago
                uint32_t mx[32];
#pragma unroll 1
                for (int ph = 0; ph < (EPI == EPI_STORE_POOL ? 5 : 4); ++ph, ++chunk_it) {
                    const uint32_t obuf = sOut + (eg * p.n_out + (chunk_it - fdiv(chunk_it, p.fd_nout) * p.fd_nout.d)) * kOutStage;
                    if (lane == 0) {
                        if (p.n_out == 3) tma_store_wait_read<2>(); else tma_store_wait_read<1>();
                    }
                    __syncwarp();
                    uint32_t pk[32];
                    if (ph < 4) {
#pragma unroll
                        for (int half = 0; half < 2; ++half) {
                            uint32_t v[32];
                            tmem_ld32(t_addr + ph * 64 + half * 32, v);
                            tmem_ld_wait();
#pragma unroll
                            for (int i = 0; i < 32; i += 2) {
                                float f0 = __uint_as_float(v[i]) + p.bias_c[half * 32 + i];
                                float f1 = __uint_as_float(v[i + 1]) + p.bias_c[half * 32 + i + 1];
                                if (p.relu) {
                                    f0 = fmaxf(f0, 0.f);
                                    f1 = fmaxf(f1, 0.f);
                                }
                                pk[half * 16 + i / 2] = pack_bf16x2(f0, f1);
                            }
                        }
                        if (ph == 3) {
                            tc_fence_before();
                            __syncwarp();
                            if (lane == 0) release_acc(acc);
                        }
                        if (EPI == EPI_STORE_POOL) {
                            // 2x2 max-pool (unet_model.py:34,57) = max over the four phases of this block position;
                            // bf16 rounding is monotone, so max of rounded == rounded max
#pragma unroll
                            for (int i = 0; i < 32; ++i) mx[i] = ph == 0 ? pk[i] : max_bf16x2(mx[i], pk[i]);
                        }
                    } else {
#pragma unroll
                        for (int i = 0; i < 32; ++i) pk[i] = mx[i];
                    }
#pragma unroll
                    for (int c16 = 0; c16 < 8; ++c16)
                        st_shared_v4(obuf + row * 128 + ((c16 ^ (row & 7)) << 4), pk[c16 * 4], pk[c16 * 4 + 1],
                                     pk[c16 * 4 + 2], pk[c16 * 4 + 3]);
                    fence_proxy_async_smem();
                    __syncwarp();
                    if (lane == 0) {
                        // this warp's four block rows: phase ph through its strided map, the pooled tile as it is
                        if (valid) tma_store_4d(ph < 4 ? &p.tmOut[ph] : &p.tmPool, obuf + q * 4096, 0, x0, y0 + 4 * q, n);
                        tma_store_commit();
                    }
                }
            }
        }
        if (EPI != EPI_HEAD && lane == 0) tma_store_wait_all<0>();
    }

    tc_fence_before();
    cluster_sync_all();
    if (warp == 2) {
        tc_fence_after();
        tmem_dealloc_pair<512>(tmem_base);
    }
}

}  // namespace ub
