// C ABI (include/unetb200.h) over the sm_100a kernels in this directory.
// Host side only builds tensor maps / launch plans and enqueues kernels; it owns
// no device memory on the hot path (see DESIGN.md, "Ownership").
#include "../../include/unetb200.h"

#include <cuda.h>
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdio>
#include <cmath>
#include <cstring>
#include <map>
#include <mutex>
#include <string>
#include <tuple>
#include <vector>

#include "conv_tc.cuh"
#include "conv_row.cuh"
#include "conv_phase.cuh"
#include "conv_phase_multi.cuh"
#include "conv_ps64.cuh"
#include "conv_phase_stack.cuh"
#include "errors.h"
#include "pack.cuh"
#include "prepost.cuh"
#include "stem.cuh"

namespace {

thread_local std::string g_err;

int fail(int code, const std::string& msg) {
    g_err = msg;
    return code;
}

}  // namespace

int ub_fail(int code, const char* msg) { return fail(code, msg); }

namespace {

#define UB_CUDA(expr)                                                                          \
    do {                                                                                       \
        cudaError_t e_ = (expr);                                                               \
        if (e_ != cudaSuccess)                                                                 \
            return fail(UNETB200_ECUDA, std::string(#expr) + ": " + cudaGetErrorString(e_));   \
    } while (0)

// ------------------------------------------------------------------ driver entry point
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*,
                                  const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                  const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn encode_tiled() {
    static EncodeTiledFn fn = nullptr;
    static std::once_flag once;
    std::call_once(once, [] {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) ==
                cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(p);
    });
    return fn;
}

// 4-D bf16 activation view: dims (C, W, H, N) with explicit byte strides for W, H, N.
int make_map4(CUtensorMap* m, const void* base, uint64_t C, uint64_t W, uint64_t H, uint64_t N,
              uint64_t strideW, uint64_t strideH, uint64_t strideN, uint32_t boxW, uint32_t boxH) {
    EncodeTiledFn enc = encode_tiled();
    if (!enc) return fail(UNETB200_ECUDA, "cuTensorMapEncodeTiled entry point unavailable");
    cuuint64_t dims[4] = {C, W, H, N};
    cuuint64_t strides[3] = {strideW, strideH, strideN};
    cuuint32_t box[4] = {64, boxW, boxH, 1};
    cuuint32_t estr[4] = {1, 1, 1, 1};
    CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(base), dims, strides,
                     box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                     CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        char buf[256];
        snprintf(buf, sizeof buf,
                 "cuTensorMapEncodeTiled(4d) failed: %d (C=%llu W=%llu H=%llu N=%llu box=%u,%u base=%p)",
                 static_cast<int>(r), (unsigned long long)C, (unsigned long long)W,
                 (unsigned long long)H, (unsigned long long)N, boxW, boxH, base);
        return fail(UNETB200_ECUDA, buf);
    }
    return 0;
}

int make_act_map(CUtensorMap* m, const void* base, int C, int W, int H, int N, int boxW, int boxH) {
    return make_map4(m, base, C, W, H, N, uint64_t(C) * 2, uint64_t(W) * C * 2,
                     uint64_t(H) * W * C * 2, boxW, boxH);
}

// weights: dims (CinTot, rows, taps)
int make_w_map(CUtensorMap* m, const void* base, int cin, int rows, int taps, int bn, int box_taps = 1) {
    EncodeTiledFn enc = encode_tiled();
    if (!enc) return fail(UNETB200_ECUDA, "cuTensorMapEncodeTiled entry point unavailable");
    cuuint64_t dims[3] = {uint64_t(cin), uint64_t(rows), uint64_t(taps)};
    cuuint64_t strides[2] = {uint64_t(cin) * 2, uint64_t(rows) * cin * 2};
    cuuint32_t box[3] = {64, uint32_t(bn), uint32_t(box_taps)};
    cuuint32_t estr[3] = {1, 1, 1};
    CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(base), dims, strides,
                     box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                     CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS)
        return fail(UNETB200_ECUDA, "cuTensorMapEncodeTiled(weights) failed: " + std::to_string(int(r)));
    return 0;
}

bool valid_x_fmt(int x_fmt) { return x_fmt >= 0 && x_fmt < ub::kNumXFormats; }

// network input of the first conv (conv_tc.cuh, A_STEM): the 18 x 10 halo patch of a tile as one TMA box
// (geometry: stem.cuh stem_box_w).
//   NCHW [N][C][H][W]      -> 4-D map (W, H, C, N), box (16 fp32 | 24 16-bit elements, 18, C, 1)
//   NHWC [N][H][W][C]      -> 3-D map (W * C, H, N), box (48 | 32 bytes for uint8, 36 | 16 fp32, 40 | 24 16-bit, 18, 1)
// The boxes are wider than the 10 columns used because a TMA tile load faults unless its innermost start
// coordinate sits on a 16-byte boundary (conv_tc.cuh).  Out-of-image elements are zero-filled, which is the conv
// padding (byte 0 -> 0 / 255; +0.0 in every float format).
int make_input_map(CUtensorMap* m, const void* x, int x_fmt, int cin, int W, int H, int N) {
    EncodeTiledFn enc = encode_tiled();
    if (!enc) return fail(UNETB200_ECUDA, "cuTensorMapEncodeTiled entry point unavailable");
    if (!valid_x_fmt(x_fmt)) return fail(UNETB200_EINVAL, "unknown x_fmt");
    if (reinterpret_cast<uintptr_t>(x) & 15) return fail(UNETB200_EINVAL, "stem: the input tensor must be 16-byte aligned");
    const uint64_t e = ub::x_elem_bytes(x_fmt);
    const CUtensorMapDataType dt = e == 4 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32
                                 : e == 1 ? CU_TENSOR_MAP_DATA_TYPE_UINT8
                                 : (x_fmt == UNETB200_X_F16_NCHW || x_fmt == UNETB200_X_F16_NHWC) ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16
                                                                                                  : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;
    const cuuint32_t bw = static_cast<cuuint32_t>(ub::stem_box_w(x_fmt, cin));
    CUresult r;
    if (!ub::x_is_nhwc(x_fmt)) {
        if ((W * e) % 16) return fail(UNETB200_EINVAL, "stem: NCHW input needs rows of a multiple of 16 bytes");
        cuuint64_t dims[4] = {uint64_t(W), uint64_t(H), uint64_t(cin), uint64_t(N)};
        cuuint64_t strides[3] = {uint64_t(W) * e, uint64_t(H) * W * e, uint64_t(cin) * H * W * e};
        cuuint32_t box[4] = {bw, 18, uint32_t(cin), 1};
        cuuint32_t estr[4] = {1, 1, 1, 1};
        r = enc(m, dt, 4, const_cast<void*>(x), dims, strides, box, estr,
                CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    } else {
        if ((W * cin * e) % 16) return fail(UNETB200_EINVAL, "stem: NHWC input needs rows of a multiple of 16 bytes");
        cuuint64_t dims[3] = {uint64_t(W) * cin, uint64_t(H), uint64_t(N)};
        cuuint64_t strides[2] = {uint64_t(W) * cin * e, uint64_t(H) * W * cin * e};
        cuuint32_t box[3] = {bw, 18, 1};
        cuuint32_t estr[3] = {1, 1, 1};
        r = enc(m, dt, 3, const_cast<void*>(x), dims, strides, box, estr,
                CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    }
    if (r != CUDA_SUCCESS)
        return fail(UNETB200_ECUDA, "cuTensorMapEncodeTiled(network input) failed: " + std::to_string(int(r)));
    return 0;
}

// ------------------------------------------------------------------ layer table
struct LayerSpec {
    const char* name;
    const char* bn;
    int kind, cin, cout, level;
};

// The stem's weight region holds two layouts: fp32 [9*cin][cout] for the CUDA-core kernel
// (stem.cuh), then bf16 hi/lo [cout][128] for the tensor-core stem (conv_tc.cuh, A_STEM).
uint64_t stem_tc_offset(int cin, int cout) { return (uint64_t(9) * cin * cout * 4 + 255) / 256 * 256; }
// ... then the smem image of the patch stem's weight tiles (A_STEMP), 9 taps x 4096 B.
uint64_t stem_patch_offset(int cin, int cout) { return stem_tc_offset(cin, cout) + uint64_t(cout) * 128 * 2; }

std::vector<unetb200_layer_t> layer_table(const unetb200_arch_t& a) {
    const int w = a.base_width;
    const LayerSpec specs[] = {
        {"down1.net.0", "down1.net.1", UNETB200_STEM, a.n_channels, w, 0},
        {"down1.net.3", "down1.net.4", UNETB200_CONV3X3, w, w, 0},
        {"down2.net.0", "down2.net.1", UNETB200_CONV3X3, w, 2 * w, 1},
        {"down2.net.3", "down2.net.4", UNETB200_CONV3X3, 2 * w, 2 * w, 1},
        {"down3.net.0", "down3.net.1", UNETB200_CONV3X3, 2 * w, 4 * w, 2},
        {"down3.net.3", "down3.net.4", UNETB200_CONV3X3, 4 * w, 4 * w, 2},
        {"down4.net.0", "down4.net.1", UNETB200_CONV3X3, 4 * w, 8 * w, 3},
        {"down4.net.3", "down4.net.4", UNETB200_CONV3X3, 8 * w, 8 * w, 3},
        {"bottleneck.net.0", "bottleneck.net.1", UNETB200_CONV3X3, 8 * w, 16 * w, 4},
        {"bottleneck.net.3", "bottleneck.net.4", UNETB200_CONV3X3, 16 * w, 16 * w, 4},
        {"up4", "", UNETB200_CONVT2X2, 16 * w, 8 * w, 4},
        {"conv4.net.0", "conv4.net.1", UNETB200_CONV3X3, 16 * w, 8 * w, 3},
        {"conv4.net.3", "conv4.net.4", UNETB200_CONV3X3, 8 * w, 8 * w, 3},
        {"up3", "", UNETB200_CONVT2X2, 8 * w, 4 * w, 3},
        {"conv3.net.0", "conv3.net.1", UNETB200_CONV3X3, 8 * w, 4 * w, 2},
        {"conv3.net.3", "conv3.net.4", UNETB200_CONV3X3, 4 * w, 4 * w, 2},
        {"up2", "", UNETB200_CONVT2X2, 4 * w, 2 * w, 2},
        {"conv2.net.0", "conv2.net.1", UNETB200_CONV3X3, 4 * w, 2 * w, 1},
        {"conv2.net.3", "conv2.net.4", UNETB200_CONV3X3, 2 * w, 2 * w, 1},
        {"up1", "", UNETB200_CONVT2X2, 2 * w, w, 1},
        {"conv1.net.0", "conv1.net.1", UNETB200_CONV3X3, 2 * w, w, 0},
        {"conv1.net.3", "conv1.net.4", UNETB200_CONV3X3, w, w, 0},
        {"out_conv", "", UNETB200_HEAD, w, a.n_classes, 0},
    };
    std::vector<unetb200_layer_t> out;
    uint64_t off = 0;
    auto align = [](uint64_t v) { return (v + 255) / 256 * 256; };
    for (const LayerSpec& s : specs) {
        unetb200_layer_t l;
        memset(&l, 0, sizeof l);
        snprintf(l.name, sizeof l.name, "%s", s.name);
        snprintf(l.bn_name, sizeof l.bn_name, "%s", s.bn);
        l.kind = s.kind;
        l.cin = s.cin;
        l.cout = s.cout;
        l.level = s.level;
        uint64_t wb = 0;
        switch (s.kind) {
            case UNETB200_STEM: wb = stem_patch_offset(s.cin, s.cout) + 9 * 4096; break;
            case UNETB200_CONV3X3: wb = uint64_t(9) * s.cin * s.cout * 2; break;
            case UNETB200_CONVT2X2: wb = uint64_t(4) * s.cin * s.cout * 2; break;
            case UNETB200_HEAD: wb = uint64_t(s.cin) * s.cout * 4; break;
        }
        l.w_off = off;
        l.w_bytes = wb;
        off = align(off + wb);
        l.b_off = off;
        l.b_bytes = uint64_t(s.cout) * 4;
        off = align(off + l.b_bytes);
        out.push_back(l);
    }
    return out;
}

// Decoder levels with the up-conv folded into the following 3x3 conv (conv_phase.cuh): level j = 1..4 is
// up{j} + conv{j}.net.0.  Their composite weights ([16][Cout][Clow] bf16) and border-case biases ([9][Cout] fp32,
// then one flag word) live behind the per-layer regions of the blob.
struct FusedUp {
    int clow, cmid, cout;          // channels of the low-resolution source, of the up-conv output (= skip), of the conv
    int li_up, li_conv;            // rows of the layer table
    uint64_t w_off, w_bytes, b_off, b_bytes, flag_off;
};

std::vector<FusedUp> fused_table(const unetb200_arch_t& a) {
    const std::vector<unetb200_layer_t> t = layer_table(a);
    const unetb200_layer_t& last = t.back();
    uint64_t off = (last.b_off + last.b_bytes + 255) / 256 * 256;
    std::vector<FusedUp> out(5);
    for (int j = 4; j >= 1; --j) {
        FusedUp f;
        f.li_up = 10 + 3 * (4 - j);
        f.li_conv = f.li_up + 1;
        f.clow = t[f.li_up].cin;
        f.cmid = t[f.li_up].cout;
        f.cout = t[f.li_conv].cout;
        f.w_off = off;
        f.w_bytes = uint64_t(16) * f.cout * f.clow * 2;
        off = (off + f.w_bytes + 255) / 256 * 256;
        f.b_off = off;
        f.b_bytes = uint64_t(9) * f.cout * 4;
        f.flag_off = f.b_off + f.b_bytes;
        off = (f.flag_off + 4 + 255) / 256 * 256;
        out[j] = f;
    }
    out[0] = FusedUp();
    out[0].w_off = off;            // end of the blob
    return out;
}

int check_arch(const unetb200_arch_t* a) {
    if (!a) return fail(UNETB200_EINVAL, "arch is NULL");
    if (a->base_width != 64) return fail(UNETB200_EINVAL, "base_width must be 64");
    if (!(a->n_channels == 1 || a->n_channels == 3 || a->n_channels == 4))
        return fail(UNETB200_EINVAL, "n_channels must be 1, 3 or 4");
    if (a->n_classes < 1 || a->n_classes > ub::kMaxClasses)
        return fail(UNETB200_EINVAL, "n_classes must be in 1..8");
    return 0;
}

// ------------------------------------------------------------------ kernel launch plumbing
typedef void (*ConvKernel)(const ub::ConvParams);

struct ConvLaunch {
    ConvKernel fn = nullptr;
    int a_stage = 0, b_stage = 0;   // bytes per activation item / weight ring stage
    int b_tap = 0, tpb = 1;         // bytes of one tap's weight tile, taps per stage (= per TMA box)
    int smem = 0;                   // dynamic shared memory of this launch (set by plan_smem)
    bool pair = false;              // launched as clusters of 2 CTAs (cta_group::2)
    bool row = false;               // conv_row_kernel (conv_row.cuh): 4 x 128 tiles, ky taps stacked along N
    bool phase = false;             // conv_phase_kernel (conv_phase.cuh): up-conv folded into the 3x3 conv
};

template <int BN, int TAPS, int AMODE, int EPI, int X = 0, bool PAIR = false, int XF = ub::X_RUNTIME,
          int LT = ub::LOGITS_F32>
ConvLaunch conv_inst() {
    ConvLaunch l;
    l.fn = ub::conv_tc_kernel<BN, TAPS, AMODE, EPI, X, PAIR, XF, LT>;
    l.a_stage = ub::ConvCfg<BN, TAPS, AMODE, PAIR>::A_STAGE;
    l.b_stage = ub::ConvCfg<BN, TAPS, AMODE, PAIR>::B_STAGE;
    l.b_tap = ub::ConvCfg<BN, TAPS, AMODE, PAIR>::B_TAP;
    l.tpb = ub::ConvCfg<BN, TAPS, AMODE, PAIR>::TPB;
    l.pair = PAIR;
    return l;
}

// CTA-pair instantiations exist for the production staging mode (A_HALO) and the up-convs.
template <int BN>
ConvLaunch pair_pick(int taps, int epi) {
    if (taps == 1) return conv_inst<BN, 1, ub::A_TAP, ub::EPI_UPSAMPLE, 0, true>();
    switch (epi) {
        case ub::EPI_STORE: return conv_inst<BN, 9, ub::A_HALO, ub::EPI_STORE, 0, true>();
        case ub::EPI_STORE_POOL: return conv_inst<BN, 9, ub::A_HALO, ub::EPI_STORE_POOL, 0, true>();
    }
    return ConvLaunch();
}

template <int BN, int AMODE>
ConvLaunch conv3_pick_epi(int epi) {
    switch (epi) {
        case ub::EPI_STORE: return conv_inst<BN, 9, AMODE, ub::EPI_STORE>();
        case ub::EPI_STORE_POOL: return conv_inst<BN, 9, AMODE, ub::EPI_STORE_POOL>();
        default: return ConvLaunch();
    }
}

// Production staging is A_HALO; A_TAP (the canonical per-tap staging) stays in every build as its cross-check.
// A_COL3 and the patch stem (A_STEMP) are measured-and-rejected alternatives: compiled only with
// -DUNETB200_TEST_VARIANTS (UNETB200_TEST_VARIANTS=1 python -m tw_invoice_unet_ocr_llm_b200.build).
template <int BN>
ConvLaunch conv3_pick_amode(int amode, int epi) {
    switch (amode) {
        case ub::A_TAP: return conv3_pick_epi<BN, ub::A_TAP>(epi);
#ifdef UNETB200_TEST_VARIANTS
        case ub::A_COL3: return conv3_pick_epi<BN, ub::A_COL3>(epi);
#endif
        case ub::A_HALO: return conv3_pick_epi<BN, ub::A_HALO>(epi);
        default: return ConvLaunch();
    }
}

// fused head (conv1.net.3 + out_conv): n_classes == 3 (the reference's configuration) has its own instantiation;
// one per logits element type
template <int AMODE, bool PAIR>
ConvLaunch head_inst(int ncls, int logits_type) {
    const bool three = ncls == 3;
    switch (logits_type) {
        case ub::LOGITS_F32:
            return three ? conv_inst<64, 9, AMODE, ub::EPI_HEAD, 3, PAIR>() : conv_inst<64, 9, AMODE, ub::EPI_HEAD, 0, PAIR>();
        case ub::LOGITS_F16:
            return three ? conv_inst<64, 9, AMODE, ub::EPI_HEAD, 3, PAIR, ub::X_RUNTIME, ub::LOGITS_F16>()
                         : conv_inst<64, 9, AMODE, ub::EPI_HEAD, 0, PAIR, ub::X_RUNTIME, ub::LOGITS_F16>();
        case ub::LOGITS_BF16:
            return three ? conv_inst<64, 9, AMODE, ub::EPI_HEAD, 3, PAIR, ub::X_RUNTIME, ub::LOGITS_BF16>()
                         : conv_inst<64, 9, AMODE, ub::EPI_HEAD, 0, PAIR, ub::X_RUNTIME, ub::LOGITS_BF16>();
    }
    return ConvLaunch();
}

template <int CIN, int XF = ub::X_RUNTIME>
ConvLaunch stem_inst() {
    ConvLaunch l;
    l.fn = ub::conv_tc_kernel<64, 1, ub::A_STEM, ub::EPI_STORE, CIN, false, XF>;
    l.a_stage = ub::ConvCfg<64, 1, ub::A_STEM>::A_STAGE;
    l.b_stage = ub::ConvCfg<64, 1, ub::A_STEM>::B_STAGE;
    l.b_tap = ub::ConvCfg<64, 1, ub::A_STEM>::B_TAP;
    return l;
}

// im2col stem: fp32 NCHW and uint8 NHWC share the run-time-format instantiation; every other format has its own
template <int CIN>
ConvLaunch stem_pick_fmt(int x_fmt) {
    switch (x_fmt) {
        case UNETB200_X_F32_NCHW:
        case UNETB200_X_U8_NHWC: return stem_inst<CIN>();
        case UNETB200_X_F16_NCHW: return stem_inst<CIN, ub::X_F16_NCHW>();
        case UNETB200_X_BF16_NCHW: return stem_inst<CIN, ub::X_BF16_NCHW>();
        case UNETB200_X_F32_NHWC: return stem_inst<CIN, ub::X_F32_NHWC>();
        case UNETB200_X_F16_NHWC: return stem_inst<CIN, ub::X_F16_NHWC>();
        case UNETB200_X_BF16_NHWC: return stem_inst<CIN, ub::X_BF16_NHWC>();
    }
    return ConvLaunch();
}

#ifdef UNETB200_TEST_VARIANTS
template <int CIN>
ConvLaunch stemp_inst() {
    ConvLaunch l;
    l.fn = ub::conv_tc_kernel<64, 9, ub::A_STEMP, ub::EPI_STORE, CIN>;
    l.a_stage = ub::ConvCfg<64, 9, ub::A_STEMP>::A_STAGE;
    l.b_stage = ub::ConvCfg<64, 9, ub::A_STEMP>::B_STAGE;
    l.b_tap = ub::ConvCfg<64, 9, ub::A_STEMP>::B_TAP;
    return l;
}
#endif

ConvLaunch pick_conv(int taps, int bn, int amode, int epi, int stem_cin = 0, int ncls = 0, bool pair = false,
                     int stem_fmt = UNETB200_X_F32_NCHW, int logits_type = ub::LOGITS_F32) {
    if (amode == ub::A_STEMP) {
#ifdef UNETB200_TEST_VARIANTS
        switch (stem_cin) {
            case 1: return stemp_inst<1>();
            case 3: return stemp_inst<3>();
            case 4: return stemp_inst<4>();
        }
#endif
        return ConvLaunch();
    }
    if (pair && amode != ub::A_STEM && amode != ub::A_STEMP && (taps == 1 || amode == ub::A_HALO)) {
        if (epi == ub::EPI_HEAD) return head_inst<ub::A_HALO, true>(ncls, logits_type);
        switch (bn) {
            case 64: return pair_pick<64>(taps, epi);
            case 128: return pair_pick<128>(taps, epi);
            case 256: return pair_pick<256>(taps, epi);
        }
        return ConvLaunch();
    }
    if (amode == ub::A_STEM) {
        switch (stem_cin) {
            case 1: return stem_pick_fmt<1>(stem_fmt);
            case 3: return stem_pick_fmt<3>(stem_fmt);
        }
        return ConvLaunch();
    }
    if (taps == 1) {
        switch (bn) {
            case 64: return conv_inst<64, 1, ub::A_TAP, ub::EPI_UPSAMPLE>();
            case 128: return conv_inst<128, 1, ub::A_TAP, ub::EPI_UPSAMPLE>();
            case 256: return conv_inst<256, 1, ub::A_TAP, ub::EPI_UPSAMPLE>();
        }
        return ConvLaunch();
    }
    if (epi == ub::EPI_HEAD) {
        switch (amode) {
            case ub::A_TAP: return head_inst<ub::A_TAP, false>(ncls, logits_type);
#ifdef UNETB200_TEST_VARIANTS
            case ub::A_COL3: return head_inst<ub::A_COL3, false>(ncls, logits_type);
#endif
            case ub::A_HALO: return head_inst<ub::A_HALO, false>(ncls, logits_type);
        }
        return ConvLaunch();
    }
    switch (bn) {
        case 64: return conv3_pick_amode<64>(amode, epi);
        case 128: return conv3_pick_amode<128>(amode, epi);
        case 256: return conv3_pick_amode<256>(amode, epi);
    }
    return ConvLaunch();
}

typedef void (*StemKernel)(const ub::StemParams);

struct Step {
    int kind = 0;              // 0 = stem, 1 = conv_tc
    StemKernel stem_fn = nullptr;   // kind 0: the CUDA-core stem instantiation (stem.cuh)
    int layer = -1;            // index into the layer table (profiling)
    ConvLaunch conv;
    ub::ConvParams cp;
    ub::StemParams sp;
    int stem_cin = 0;
    int pdl = 0;               // launch with programmatic stream serialization
    dim3 grid, block;
};

// Describes one tensor-core conv launch; shared by the forward plan and the test hooks.
struct ConvDesc {
    const void* src0 = nullptr;
    int c0 = 0;
    const void* src1 = nullptr;
    int c1 = 0;
    const void* w = nullptr;
    const float* bias = nullptr;
    int n = 0, h = 0, wd = 0, cout = 0, relu = 1;
    int taps = 9;               // 9 = conv3x3, 1 = convT2x2
    int epi = ub::EPI_STORE;
    void* out = nullptr;
    void* pool = nullptr;
    const float* head_w = nullptr;
    const float* head_b = nullptr;
    int ncls = 0;
    void* logits = nullptr;
    int logits_type = ub::LOGITS_F32;   // element type of `logits` (UNETB200_LOGITS_*)
    uint8_t* mask = nullptr;
    int mask_bits = 0;          // 1 = mask is bit-packed [N][ncls][H][W/8]
    int bn = 128, amode = ub::A_COL3;
    int wstat = 1;              // allow weight-stationary mode when it fits
    int pf_items = 0;           // L2 prefetch distance (activation ring items)
    int epi2 = 1;               // two epilogue groups: 0 never, 1 weight-stationary launches, 2 always
    int min_na = 3;             // weight-stationary launches: activation stages wanted before staging slots
    int pair = 0;               // CTA pairs (cta_group::2) where an instantiation exists
    int fill_sms = 0;           // small batches: narrow the column block until the tiles cover the SMs
    const void* stem_x = nullptr;   // A_STEM: network input, its format and channel count
    int stem_fmt = 0, stem_cin = 0;
    int* dbg = nullptr;
};

// Shared-memory carve-up of one launch: [A ring][B ring or resident slab][out staging][pool
// staging][barriers].  Weight-stationary when the layer has one column block and its whole
// weight slab fits beside at least two activation stages.
int plan_smem(ConvLaunch* cl, ub::ConvParams* p, int taps, int n_cs, int n_blocks, int bn, bool pool,
              bool has_out, int allow_wstat, int patch_bytes, int epi2, int min_na) {
    const int budget = ub::kSmemLimit - ub::kStaticSmem - 1024 /*alignment slack*/ - patch_bytes;
    const int slab = taps * n_cs * cl->b_tap;
    // Epilogue groups: thin-K launches with resident weights are epilogue-bound -> two groups on
    // alternate tiles, two staging slots each; everything else keeps one group with two slots.
    const int slot = ub::kOutStage + (pool ? ub::kPoolStage : 0);
    int n_out = has_out ? 2 : 0, n_epi = 1, na = 0, nb = 0, wstat = 0;
    if (allow_wstat && n_blocks == 1) {
        for (int want_na = (min_na > 2 ? min_na : 2); want_na >= 2 && !wstat; --want_na) {
            for (int ne = (epi2 >= 1 ? 2 : 1); ne >= 1 && !wstat; --ne) {
                for (int no = has_out ? 2 : 0; no >= (has_out ? 1 : 0) && !wstat; --no) {
                    const int rest = budget - ub::kBarBytes - ne * no * slot - slab;
                    if (rest >= want_na * cl->a_stage) {
                        wstat = 1;
                        n_out = no;
                        n_epi = ne;
                        nb = taps * n_cs;        // (in units of one tap's tile)
                        na = rest / cl->a_stage;
                    }
                }
            }
        }
    }
    if (!wstat) {
        // weight ring: ~96 / 80 / 64 KB for BN = 256 / 128 / 64 (a CTA pair stages half rows -> twice the depth)
        nb = (bn == 256 ? 3 * 32768 : (bn == 128 ? 5 * 16384 : 8 * 8192)) / cl->b_stage;
        if (nb > ub::kMaxRing) nb = ub::kMaxRing;
        n_epi = epi2 >= 2 ? 2 : 1;
        n_out = has_out ? (n_epi == 2 ? 1 : 2) : 0;
        const int rest = budget - ub::kBarBytes - n_epi * n_out * slot - nb * cl->b_stage;
        na = rest / cl->a_stage;
    }
    if (na > ub::kMaxRing) na = ub::kMaxRing;
    if (patch_bytes && !wstat) return fail(UNETB200_EINVAL, "stem: weights must be resident");
    if (na < 2) return fail(UNETB200_EINVAL, "conv: shared memory plan does not fit");
    p->na = na;
    p->nb = nb;
    p->wstat = wstat;
    p->n_out = n_out ? n_out : 1;
    p->off_b = na * cl->a_stage;
    p->off_out = p->off_b + (wstat ? slab : nb * cl->b_stage);
    p->n_epi = n_epi;
    p->off_pool = p->off_out + n_epi * n_out * ub::kOutStage;
    p->off_bar = p->off_pool + (pool ? n_epi * n_out * ub::kPoolStage : 0);
    p->off_patch = p->off_bar + ub::kBarBytes;
    cl->smem = p->off_patch + patch_bytes + 1024;
    return 0;
}

// Row-stacked kernel for the 64-output-channel 3x3 convs (conv_row.cuh).
int build_row_step(const ConvDesc& d, int num_sms, Step* st) {
    if (d.taps != 9 || d.cout != 64) return fail(UNETB200_EINVAL, "row kernel: 3x3 conv with 64 output channels only");
    if (d.c0 <= 0 || d.c0 % 64 || d.c1 % 64 || d.c1 < 0)
        return fail(UNETB200_EINVAL, "conv: source channels must be multiples of 64");
    const int n_cs = (d.c0 + d.c1) / 64;
    st->kind = 1;
    ConvLaunch& cl = st->conv;
    cl = ConvLaunch();
    cl.row = true;
    switch (d.epi) {
        case ub::EPI_STORE: cl.fn = ub::conv_row_kernel<ub::EPI_STORE>; break;
        case ub::EPI_STORE_POOL: cl.fn = ub::conv_row_kernel<ub::EPI_STORE_POOL>; break;
        case ub::EPI_HEAD:
            switch (d.logits_type) {
                case ub::LOGITS_F32: cl.fn = d.ncls == 3 ? ub::conv_row_kernel<ub::EPI_HEAD, 3> : ub::conv_row_kernel<ub::EPI_HEAD, 0>; break;
                case ub::LOGITS_F16:
                    cl.fn = d.ncls == 3 ? ub::conv_row_kernel<ub::EPI_HEAD, 3, ub::LOGITS_F16> : ub::conv_row_kernel<ub::EPI_HEAD, 0, ub::LOGITS_F16>;
                    break;
                case ub::LOGITS_BF16:
                    cl.fn = d.ncls == 3 ? ub::conv_row_kernel<ub::EPI_HEAD, 3, ub::LOGITS_BF16> : ub::conv_row_kernel<ub::EPI_HEAD, 0, ub::LOGITS_BF16>;
                    break;
                default: return fail(UNETB200_EINVAL, "unknown logits_type");
            }
            break;
        default: return fail(UNETB200_EINVAL, "row kernel: unsupported epilogue");
    }
    ub::ConvParams& p = st->cp;
    memset(&p, 0, sizeof p);
    int rc;
    if ((rc = make_act_map(&p.tmA0, d.src0, d.c0, d.wd, d.h, d.n, ub::kRowW + 2, 1))) return rc;
    if (d.c1 > 0) {
        if ((rc = make_act_map(&p.tmA1, d.src1, d.c1, d.wd, d.h, d.n, ub::kRowW + 2, 1))) return rc;
    } else {
        p.tmA1 = p.tmA0;
    }
    if ((rc = make_w_map(&p.tmB, d.w, d.c0 + d.c1, 64, 9, 64, 1))) return rc;
    if (d.epi != ub::EPI_HEAD) {
        if ((rc = make_act_map(&p.tmOut[0], d.out, 64, d.wd, d.h, d.n, 32, 1))) return rc;   // one warp's 32 pixels of a row
        for (int i = 1; i < 4; ++i) p.tmOut[i] = p.tmOut[0];
    }
    if (d.epi == ub::EPI_STORE_POOL) {
        if (!d.pool) return fail(UNETB200_EINVAL, "pool output missing");
        if ((rc = make_act_map(&p.tmPool, d.pool, 64, d.wd / 2, d.h / 2, d.n, 16, 1))) return rc;
    } else {
        p.tmPool = p.tmA0;
    }
    p.bias = d.bias; p.head_w = d.head_w; p.head_b = d.head_b; p.logits = d.logits; p.mask = d.mask;
    p.mask_bits = d.mask_bits; p.dbg = d.dbg;
    // bias / head weights travel as kernel parameters (constant bank): one small synchronous read-back per plan
    UB_CUDA(cudaMemcpy(p.bias_c, d.bias, sizeof p.bias_c, cudaMemcpyDeviceToHost));
    if (d.epi == ub::EPI_HEAD) {
        if (!d.head_w || !d.head_b || d.ncls < 1 || d.ncls > ub::kMaxClasses)
            return fail(UNETB200_EINVAL, "row kernel: head weights missing");
        UB_CUDA(cudaMemcpy(p.head_wc, d.head_w, sizeof(float) * 64 * d.ncls, cudaMemcpyDeviceToHost));
        UB_CUDA(cudaMemcpy(p.head_bc, d.head_b, sizeof(float) * d.ncls, cudaMemcpyDeviceToHost));
    }
    p.C0 = d.c0; p.C1 = d.c1; p.H = d.h; p.W = d.wd; p.NIMG = d.n; p.Cout = 64;
    p.tiles_x = (d.wd + ub::kRowW - 1) / ub::kRowW;
    p.tiles_y = (d.h + ub::kRowR - 1) / ub::kRowR;
    p.n_blocks = 1;
    const long long total = 1LL * p.tiles_x * p.tiles_y * d.n;
    if (total > 0x7fffffffLL) return fail(UNETB200_EINVAL, "conv: too many tiles");
    p.total_tiles = static_cast<int>(total);
    p.relu = d.relu; p.ncls = d.ncls; p.wstat = 1;
    // shared memory: [A ring][resident weights][row staging][pool staging][barriers]
    const int budget = ub::kSmemLimit - ub::kRowStatic - 1024 /*alignment slack*/ - ub::kBarBytes;
    const int slab = n_cs * 9 * ub::kRowBBlock;
    int n_epi = 2, n_out = 0, pool_bytes = 0;
    if (d.epi == ub::EPI_STORE) n_out = 2;
    if (d.epi == ub::EPI_STORE_POOL) { n_out = 2; pool_bytes = 8192; }          // two rows + one pooled row per group
    auto staging = [&]() { return n_epi * (n_out * ub::kOutStage + pool_bytes); };
    // prefer activation ring depth over staging: at least 4 halo rows in flight
    while (d.epi == ub::EPI_STORE && (budget - slab - staging()) / ub::kRowAStage < 4 && (n_out > 1 || n_epi > 1)) {
        if (n_out > 1) n_out = 1; else n_epi = 1;
    }
    while (d.epi == ub::EPI_STORE_POOL && (budget - slab - staging()) / ub::kRowAStage < 4 && n_epi > 1) n_epi = 1;
    int na = (budget - slab - staging()) / ub::kRowAStage;
    if (na > ub::kMaxRing) na = ub::kMaxRing;
    if (na < 2) return fail(UNETB200_EINVAL, "row kernel: shared memory plan does not fit");
    p.na = na; p.nb = n_cs * 9; p.n_out = n_out ? n_out : 1; p.n_epi = n_epi;
    p.off_b = na * ub::kRowAStage;
    p.off_out = p.off_b + slab;
    p.off_pool = p.off_out + n_epi * n_out * ub::kOutStage;
    p.off_bar = p.off_pool + n_epi * pool_bytes;
    cl.smem = p.off_bar + ub::kBarBytes + 1024;
    cl.a_stage = ub::kRowAStage; cl.b_tap = ub::kRowBBlock; cl.b_stage = ub::kRowBBlock;
    p.fd_tpi = ub::make_fastdiv(static_cast<uint32_t>(p.tiles_x * p.tiles_y));
    p.fd_tx = ub::make_fastdiv(static_cast<uint32_t>(p.tiles_x));
    p.fd_nb = ub::make_fastdiv(1u);
    p.fd_na = ub::make_fastdiv(static_cast<uint32_t>(na));
    p.fd_nout = ub::make_fastdiv(static_cast<uint32_t>(p.n_out));
    st->grid = dim3(static_cast<unsigned>(total < num_sms ? total : num_sms));
    st->block = dim3(384);
    return 0;
}

// ConvTranspose2d(2,2) + 3x3 conv over cat([up, skip]) as ONE launch (conv_phase.cuh).
struct PhaseDesc {
    const void* low = nullptr;      // low-resolution source [N][h][w][c_low] bf16
    int c_low = 0;
    const void* skip = nullptr;     // skip tensor [N][2h][2w][c_skip] bf16
    int c_skip = 0;
    const void* wc = nullptr;       // composite weights [16][cout][c_low] bf16 (pack_fused_up_w_kernel)
    const void* w3 = nullptr;       // the 3x3 conv's packed weights [9][cout][c_up + c_skip] bf16
    int c_up = 0;                   // K columns of the up half in w3
    const float* bias9 = nullptr;   // [9][cout]
    int n = 0, h = 0, wd = 0;       // LOW-resolution size
    int cout = 0, relu = 1;
    void* out = nullptr;            // [N][2h][2w][cout] bf16
    int bn = 256, pair = 1;
    int one_phase = 0;              // 1 = one phase per unit whatever the column block (cross-check / A-B variant)
    int stack = 0;                  // 1 = phase-stacked kernel (conv_phase_stack.cuh) where it applies: 64 output and 64 skip channels, CTA pairs
    int fill_sms = 0;               // small batches: 128-column blocks on the one-phase kernel when 256-column units do not cover the SMs
    int* dbg = nullptr;
};

// one phase per work unit (conv_phase.cuh)
template <int BN>
void phase_inst(bool pair, ConvLaunch* cl, int* box_w, int* box_h, int* nph) {
    cl->fn = pair ? ub::conv_phase_kernel<BN, true> : ub::conv_phase_kernel<BN, false>;
    cl->a_stage = ub::kPhAStage;
    *box_w = ub::kPhBoxW;
    *box_h = ub::kPhBoxH;
    *nph = 1;
}
// NPY x NPX phases per work unit (conv_phase_multi.cuh)
template <int BN, int NPY, int NPX>
void phase_multi_inst(bool pair, ConvLaunch* cl, int* box_w, int* box_h, int* nph) {
    cl->fn = pair ? ub::conv_phase_multi_kernel<BN, true, NPY, NPX> : ub::conv_phase_multi_kernel<BN, false, NPY, NPX>;
    cl->a_stage = ub::PhaseMultiCfg<BN, true, NPY, NPX>::A_STAGE;
    *box_w = ub::PhaseMultiCfg<BN, true, NPY, NPX>::BW;
    *box_h = ub::PhaseMultiCfg<BN, true, NPY, NPX>::BH;
    *nph = NPY * NPX;
}

int build_phase_step(const PhaseDesc& d, int num_sms, Step* st) {
    if (d.c_low <= 0 || d.c_low % 64 || d.c_skip <= 0 || d.c_skip % 64 || d.cout % 64 || d.cout <= 0 || d.c_up % 64)
        return fail(UNETB200_EINVAL, "fused up-conv: channel counts must be multiples of 64");
    if (d.cout > 512) return fail(UNETB200_EINVAL, "fused up-conv: at most 512 output channels");
    int bn = d.bn;
    if (bn > d.cout) bn = d.cout;
    while (d.cout % bn) bn >>= 1;
    if (!(bn == 64 || bn == 128 || bn == 256)) return fail(UNETB200_EINVAL, "fused up-conv: bad column block");
    const bool pair = d.pair != 0;
    // Batch-1 latency (BASELINE configs[4]), as in build_conv_step: the deepest folded level has 8 tile positions per
    // image, so its 256-column units (4 phases x 2 blocks x 4 pairs = 32) leave most SMs idle; the SAME one-phase kernel
    // with 128-column blocks has twice the units at a lower tensor-pipe rate (0.70 vs 0.985, profiles/) and the same K
    // order per output element -> same bits.  Larger batches keep the wide blocks.
    bool narrow = false;
    if (d.fill_sms && bn == 256 && !d.one_phase && d.cout % 128 == 0) {
        const long long mt = 1LL * ((d.wd + 7) / 8) * ((d.h + 15) / 16) * d.n;
        const long long mu = pair ? (mt + 1) / 2 : mt;
        const long long slots = pair ? num_sms / 2 : num_sms;
        auto cost = [&](int b, double eff) {
            const long long units = mu * 4 * (d.cout / b);
            return static_cast<double>((units + slots - 1) / slots) * b / eff;
        };
        if (cost(128, 0.70) < 0.97 * cost(256, 0.985)) { bn = 128; narrow = true; }
    }
    st->kind = 1;
    ConvLaunch& cl = st->conv;
    cl = ConvLaunch();
    cl.phase = true;
    cl.pair = pair;
    // phases per work unit: 1 for 256-column blocks (conv_phase.cuh), px = 0, 1 side by side for 128, all four for 64
    // (conv_phase_multi.cuh); one_phase forces the one-phase kernel (cross-check / A-B)
    int box_w = 0, box_h = 0, nph = 1;
    if (bn == 256) phase_inst<256>(pair, &cl, &box_w, &box_h, &nph);
    else if (bn == 128 && (d.one_phase || narrow)) phase_inst<128>(pair, &cl, &box_w, &box_h, &nph);
    else if (bn == 128) phase_multi_inst<128, 1, 2>(pair, &cl, &box_w, &box_h, &nph);
    else if (d.one_phase) phase_inst<64>(pair, &cl, &box_w, &box_h, &nph);
    else phase_multi_inst<64, 2, 2>(pair, &cl, &box_w, &box_h, &nph);
    // phase-stacked form of the 2 x 2 kernel (conv_phase_stack.cuh): resident skip-half images, CTA-specific stages
    const bool stack = d.stack && bn == 64 && pair && !d.one_phase && d.cout == 64 && d.c_skip == 64;
    if (stack) {
        cl.fn = ub::conv_phase_stack64_kernel;
        cl.a_stage = ub::kPsSlot;
        box_w = ub::kPsBoxW; box_h = ub::kPsBoxH; nph = 4;
    }
    cl.b_tap = (pair ? bn / 2 : bn) * 128;
    const bool multi = nph > 1;                  // conv_phase_multi.cuh: weight stages of 4 composite / 3 skip taps
    cl.b_stage = multi ? 4 * cl.b_tap : cl.b_tap;
    ub::ConvParams& p = st->cp;
    memset(&p, 0, sizeof p);
    int rc;
    const int ho = 2 * d.h, wo = 2 * d.wd;
    if ((rc = make_act_map(&p.tmA0, d.low, d.c_low, d.wd, d.h, d.n, box_w, box_h))) return rc;
    p.tmA1 = p.tmA0;
    p.tmPool = p.tmA0;
    for (int q = 0; q < 4; ++q) {
        const int qy = q >> 1, qx = q & 1;
        // parity plane (qy, qx) of the skip tensor / of the output: pixel (i, j) of the plane is (2i + qy, 2j + qx)
        const char* sb = static_cast<const char*>(d.skip) + (uint64_t(qy) * wo + qx) * d.c_skip * 2;
        if ((rc = make_map4(&p.tmP[q], sb, d.c_skip, d.wd, d.h, d.n, uint64_t(2) * d.c_skip * 2,
                            uint64_t(2) * wo * d.c_skip * 2, uint64_t(ho) * wo * d.c_skip * 2, box_w, box_h)))
            return rc;
        const char* ob = static_cast<const char*>(d.out) + (uint64_t(qy) * wo + qx) * d.cout * 2;
        if ((rc = make_map4(&p.tmOut[q], ob, d.cout, d.wd, d.h, d.n, uint64_t(2) * d.cout * 2,
                            uint64_t(2) * wo * d.cout * 2, uint64_t(ho) * wo * d.cout * 2, 8, 4)))
            return rc;
    }
    if ((rc = make_w_map(&p.tmB, d.wc, d.c_low, d.cout, 16, pair ? bn / 2 : bn, multi ? 4 : 1))) return rc;
    if ((rc = make_w_map(&p.tmB2, d.w3, d.c_up + d.c_skip, d.cout, 9, pair ? bn / 2 : bn, multi ? 3 : 1))) return rc;
    p.tmB3 = p.tmB2; p.tmB4 = p.tmB2;
    if (stack) {
        if ((rc = make_w_map(&p.tmB, d.wc, d.c_low, 64, 16, 64, 1))) return rc;
        if ((rc = make_w_map(&p.tmB2, d.wc, d.c_low, 64, 16, 32, 1))) return rc;
        if ((rc = make_w_map(&p.tmB3, d.w3, d.c_up + d.c_skip, 64, 9, 64, 1))) return rc;
        if ((rc = make_w_map(&p.tmB4, d.w3, d.c_up + d.c_skip, 64, 9, 32, 1))) return rc;
        // the interior border case (row 4 of bias9) as kernel parameters: constant-bank operands of the epilogue's FADDs
        UB_CUDA(cudaMemcpy(p.bias_c, d.bias9 + 4 * 64, sizeof p.bias_c, cudaMemcpyDeviceToHost));
    }
    p.bias9 = d.bias9;
    p.kskip = d.c_up;
    p.dbg = d.dbg;
    p.C0 = d.c_low; p.C1 = d.c_skip; p.H = d.h; p.W = d.wd; p.NIMG = d.n; p.Cout = d.cout;
    p.tiles_x = (d.wd + 7) / 8;
    p.tiles_y = (d.h + 15) / 16;
    p.n_blocks = d.cout / bn;
    const long long m_tiles = 1LL * p.tiles_x * p.tiles_y * d.n;
    const long long units = (pair ? (m_tiles + 1) / 2 : m_tiles) * (4 / nph) * p.n_blocks;
    if (units > 0x7fffffffLL) return fail(UNETB200_EINVAL, "conv: too many tiles");
    p.total_tiles = static_cast<int>(m_tiles * 4 * p.n_blocks);
    p.relu = d.relu;
    // shared memory: [A ring][B ring][out staging][barriers][bias9]
    const int bias_bytes = (9 * d.cout * 4 + 1023) / 1024 * 1024;
    const int budget = ub::kSmemLimit - ub::kRowStatic - 1024 /*alignment slack*/ - bias_bytes - ub::kBarBytes;   // (no static shared memory)
    int nb = (bn == 256 ? 3 * 32768 : (bn == 128 ? 5 * 16384 : 8 * 8192)) / cl.b_stage;
    if (multi) nb = (bn == 128 ? 98304 : 65536) / cl.b_stage;   // 96 / 64 KB of weight stages (pairs: 3 / 4 stages), the rest is activation slots (one box each)
    if (multi && nb < 2) nb = 2;
    if (nb > ub::kMaxRing) nb = ub::kMaxRing;
    // stacked: [A ring][up-half stages][resident skip images 72 KB][staging]: three stages leave three box slots
    const int resident = stack ? ub::kPsWBytes : 0;
    if (stack) nb = 3;
    int n_out = 2;
    const int n_epi = 1;
    int na = (budget - n_epi * n_out * ub::kOutStage - nb * cl.b_stage - resident) / cl.a_stage;
    if (na < 3) {                                // (the unpaired cross-check variants: full-height weight stages)
        n_out = 1;
        na = (budget - n_epi * n_out * ub::kOutStage - nb * cl.b_stage - resident) / cl.a_stage;
    }
    if (na > ub::kMaxRing) na = ub::kMaxRing;
    if (na < (multi ? 3 : 2)) return fail(UNETB200_EINVAL, "fused up-conv: shared memory plan does not fit");
    p.na = na; p.nb = nb; p.wstat = 0; p.n_out = n_out; p.n_epi = n_epi;
    p.off_b = na * cl.a_stage;
    p.off_out = p.off_b + nb * cl.b_stage + resident;
    p.off_pool = p.off_out + n_epi * n_out * ub::kOutStage;
    p.off_bar = p.off_pool;
    if (stack) p.off_pool = p.off_b + nb * cl.b_stage;      // (the resident images' offset in this kernel)
    p.off_patch = p.off_bar + ub::kBarBytes;
    cl.smem = p.off_patch + bias_bytes + 1024;
    p.fd_tpi = ub::make_fastdiv(static_cast<uint32_t>(p.tiles_x * p.tiles_y));
    p.fd_tx = ub::make_fastdiv(static_cast<uint32_t>(p.tiles_x));
    p.fd_nb = ub::make_fastdiv(static_cast<uint32_t>(p.n_blocks));
    p.fd_na = ub::make_fastdiv(static_cast<uint32_t>(na));
    p.fd_nout = ub::make_fastdiv(static_cast<uint32_t>(n_out));
    if (pair) {
        const long long pairs = units < num_sms / 2 ? units : num_sms / 2;
        st->grid = dim3(static_cast<unsigned>(2 * pairs));
    } else {
        st->grid = dim3(static_cast<unsigned>(units < num_sms ? units : num_sms));
    }
    st->block = dim3(stack ? 256 : 384);         // (the stacked kernel has one epilogue group: 8 warps)
    return 0;
}

// Phase-stacked kernel for the 64 -> 64 channel 3x3 convs (conv_ps64.cuh).
int build_ps64_step(const ConvDesc& d, int num_sms, Step* st) {
    if (d.taps != 9 || d.cout != 64 || d.c0 != 64 || d.c1 != 0)
        return fail(UNETB200_EINVAL, "phase-stacked kernel: 3x3 conv, 64 -> 64 channels, one source only");
    if (d.h % 2 || d.wd % 2) return fail(UNETB200_EINVAL, "phase-stacked kernel: even H and W only");
    st->kind = 1;
    ConvLaunch& cl = st->conv;
    cl = ConvLaunch();
    cl.phase = true;            // (no static shared memory: same dynamic limit as the folded up-conv kernels)
    cl.pair = true;
    switch (d.epi) {
        case ub::EPI_STORE: cl.fn = ub::conv_ps64_kernel<ub::EPI_STORE>; break;
        case ub::EPI_STORE_POOL: cl.fn = ub::conv_ps64_kernel<ub::EPI_STORE_POOL>; break;
        case ub::EPI_HEAD:
            switch (d.logits_type) {
                case ub::LOGITS_F32: cl.fn = d.ncls == 3 ? ub::conv_ps64_kernel<ub::EPI_HEAD, 3> : ub::conv_ps64_kernel<ub::EPI_HEAD, 0>; break;
                case ub::LOGITS_F16:
                    cl.fn = d.ncls == 3 ? ub::conv_ps64_kernel<ub::EPI_HEAD, 3, ub::LOGITS_F16> : ub::conv_ps64_kernel<ub::EPI_HEAD, 0, ub::LOGITS_F16>;
                    break;
                case ub::LOGITS_BF16:
                    cl.fn = d.ncls == 3 ? ub::conv_ps64_kernel<ub::EPI_HEAD, 3, ub::LOGITS_BF16> : ub::conv_ps64_kernel<ub::EPI_HEAD, 0, ub::LOGITS_BF16>;
                    break;
                default: return fail(UNETB200_EINVAL, "unknown logits_type");
            }
            break;
        default: return fail(UNETB200_EINVAL, "phase-stacked kernel: unsupported epilogue");
    }
    ub::ConvParams& p = st->cp;
    memset(&p, 0, sizeof p);
    int rc;
    const int hb = d.h / 2, wb = d.wd / 2;      // block positions (I, J): pixel (2I + py, 2J + px)
    for (int q = 0; q < 4; ++q) {
        const int qy = q >> 1, qx = q & 1;
        const char* sb = static_cast<const char*>(d.src0) + (uint64_t(qy) * d.wd + qx) * 64 * 2;
        if ((rc = make_map4(&p.tmP[q], sb, 64, wb, hb, d.n, uint64_t(2) * 64 * 2, uint64_t(2) * d.wd * 64 * 2,
                            uint64_t(d.h) * d.wd * 64 * 2, ub::kPsBoxW, ub::kPsBoxH)))
            return rc;
        if (d.epi != ub::EPI_HEAD) {
            const char* ob = static_cast<const char*>(d.out) + (uint64_t(qy) * d.wd + qx) * 64 * 2;
            if ((rc = make_map4(&p.tmOut[q], ob, 64, wb, hb, d.n, uint64_t(2) * 64 * 2, uint64_t(2) * d.wd * 64 * 2,
                                uint64_t(d.h) * d.wd * 64 * 2, 8, 4)))
                return rc;
        } else {
            p.tmOut[q] = p.tmP[q];
        }
    }
    p.tmA0 = p.tmP[0];
    p.tmA1 = p.tmP[0];
    if ((rc = make_w_map(&p.tmB, d.w, 64, 64, 9, 64, 1))) return rc;      // image 1: whole taps
    if ((rc = make_w_map(&p.tmB2, d.w, 64, 64, 9, 32, 1))) return rc;     // image 2: half taps
    if (d.epi == ub::EPI_STORE_POOL) {
        if (!d.pool) return fail(UNETB200_EINVAL, "pool output missing");
        if ((rc = make_act_map(&p.tmPool, d.pool, 64, wb, hb, d.n, 8, 4))) return rc;
    } else {
        p.tmPool = p.tmP[0];
    }
    p.bias = d.bias; p.head_w = d.head_w; p.head_b = d.head_b; p.logits = d.logits; p.mask = d.mask;
    p.mask_bits = d.mask_bits; p.dbg = d.dbg;
    UB_CUDA(cudaMemcpy(p.bias_c, d.bias, sizeof p.bias_c, cudaMemcpyDeviceToHost));
    if (d.epi == ub::EPI_HEAD) {
        if (!d.head_w || !d.head_b || d.ncls < 1 || d.ncls > ub::kMaxClasses)
            return fail(UNETB200_EINVAL, "phase-stacked kernel: head weights missing");
        UB_CUDA(cudaMemcpy(p.head_wc, d.head_w, sizeof(float) * 64 * d.ncls, cudaMemcpyDeviceToHost));
        UB_CUDA(cudaMemcpy(p.head_bc, d.head_b, sizeof(float) * d.ncls, cudaMemcpyDeviceToHost));
    }
    p.C0 = 64; p.C1 = 0; p.H = d.h; p.W = d.wd; p.NIMG = d.n; p.Cout = 64;
    p.tiles_x = (wb + 7) / 8;
    p.tiles_y = (hb + 15) / 16;
    p.n_blocks = 1;
    const long long m_tiles = 1LL * p.tiles_x * p.tiles_y * d.n;
    if (m_tiles > 0x3fffffffLL) return fail(UNETB200_EINVAL, "conv: too many tiles");
    p.total_tiles = static_cast<int>(m_tiles);
    p.relu = d.relu; p.ncls = d.ncls; p.wstat = 1;
    // shared memory: [plane-box slots][resident weight images][staging: 3 x 16 KB per epilogue group][barriers]
    // epilogue groups alternate units; the store epilogues stage through n_out slots of 16 KB per group
    // (store epilogues: one group with three slots and more plane-box slots measured better than two groups with two
    // slots each -- ncu: down1.net.3 0.910 ms / 83.6 % tensor pipe vs 0.921 ms / 79.2 %; two groups with epi2 = 2)
    const int n_epi = (d.epi == ub::EPI_HEAD || d.epi2 >= 2) ? 2 : 1;
    const int n_out = n_epi == 2 ? 2 : 3;
    const int staging = d.epi == ub::EPI_HEAD ? 0 : n_epi * n_out * ub::kOutStage;
    const int budget = ub::kSmemLimit - ub::kPsStatic - 1024 /*alignment slack*/ - ub::kBarBytes;
    int na = (budget - ub::kPsWBytes - staging) / ub::kPsSlot;
    if (na > ub::kMaxRing) na = ub::kMaxRing;
    if (na < 2) return fail(UNETB200_EINVAL, "phase-stacked kernel: shared memory plan does not fit");
    p.na = na; p.nb = 12; p.n_out = n_out; p.n_epi = n_epi;
    p.off_b = na * ub::kPsSlot;
    p.off_out = p.off_b + ub::kPsWBytes;
    p.off_pool = p.off_out + staging;
    p.off_bar = p.off_pool;
    cl.smem = p.off_bar + ub::kBarBytes + 1024;
    cl.a_stage = ub::kPsSlot; cl.b_tap = 8192; cl.b_stage = 8192;
    p.fd_tpi = ub::make_fastdiv(static_cast<uint32_t>(p.tiles_x * p.tiles_y));
    p.fd_tx = ub::make_fastdiv(static_cast<uint32_t>(p.tiles_x));
    p.fd_nb = ub::make_fastdiv(1u);
    p.fd_na = ub::make_fastdiv(static_cast<uint32_t>(na));
    p.fd_nout = ub::make_fastdiv(static_cast<uint32_t>(n_out));
    const long long units = (m_tiles + 1) / 2;
    const long long pairs = units < num_sms / 2 ? units : num_sms / 2;
    st->grid = dim3(static_cast<unsigned>(2 * pairs));
    st->block = dim3(384);
    return 0;
}

int build_conv_step(const ConvDesc& d, int num_sms, Step* st) {
    if (d.amode == ub::A_ROW) return build_row_step(d, num_sms, st);
    if (d.amode == ub::A_PS64) return build_ps64_step(d, num_sms, st);
    const bool stemp = d.amode == ub::A_STEMP;
    const bool stem = d.amode == ub::A_STEM || stemp;
    if (d.c0 <= 0 || d.c0 % 64 || d.c1 % 64 || d.c1 < 0)
        return fail(UNETB200_EINVAL, "conv: source channels must be multiples of 64");
    if (stem && (d.taps != (stemp ? 9 : 1) || d.cout != 64 || d.c0 != 64 || d.c1 != 0 || !d.stem_x ||
                 d.epi != ub::EPI_STORE))
        return fail(UNETB200_EINVAL, "stem: bad configuration");
    if (d.cout % 64) return fail(UNETB200_EINVAL, "conv: cout must be a multiple of 64");
    const int cols = (d.taps == 1 && !stem) ? 4 * d.cout : d.cout;
    int bn = d.bn;
    if (d.epi == ub::EPI_HEAD) bn = 64;
    if (bn > cols) bn = cols;
    while (cols % bn) bn >>= 1;
    if (d.fill_sms && !stem && (d.taps == 9 || d.fill_sms > 1) && d.epi != ub::EPI_HEAD) {
        // Batch-1 latency (BASELINE configs[4]): the deep layers have few pixel tiles (32x32 pixels = 8), so
        // 256-wide column blocks leave most SMs idle; a narrower block runs each CTA at a lower tensor-pipe
        // rate (more A re-reads) but on up to 4x as many SMs.  Same K order per output -> same bits.
        // Measured (tools/ab.py fill_sms=0,1): batch 1 0.472 -> 0.393 ms (bottleneck.net.3 53 -> 29 us),
        // batch 2 / 3 / 8 -4 / -5 / -2.5 %, batch >= 16 unchanged; the up-convs (epilogue-bound scatter)
        // got slower with narrow blocks and keep theirs.
        const long long m_tiles = 1LL * ((d.wd + 7) / 8) * ((d.h + 15) / 16) * d.n;
        const bool paired = d.pair != 0 && (d.taps == 1 || d.amode == ub::A_HALO);
        const long long m_units = paired ? (m_tiles + 1) / 2 : m_tiles;
        const long long slots = paired ? num_sms / 2 : num_sms;
        // cost of a launch ~ waves x (columns per unit / tensor-pipe efficiency of that block width);
        // efficiencies as measured at batch 64 (profiles/): 0.97 / 0.95 / 0.70 for 256 / 128 / 64 columns
        auto cost = [&](int b) {
            const long long units = m_units * (cols / b);
            const long long waves = (units + slots - 1) / slots;
            return static_cast<double>(waves) * b / (b == 256 ? 0.97 : (b == 128 ? 0.95 : 0.70));
        };
        int best = bn;
        for (int b = bn >> 1; b >= 64; b >>= 1)
            if (cols % b == 0 && cost(b) < 0.97 * cost(best)) best = b;     // near ties keep the wider block
        bn = best;
    }
    if (!(bn == 64 || bn == 128 || bn == 256)) return fail(UNETB200_EINVAL, "conv: bad column block");
    if (d.epi == ub::EPI_HEAD && d.cout != 64)
        return fail(UNETB200_EINVAL, "fused head needs cout == 64");
    st->kind = 1;
    if (d.logits_type != ub::LOGITS_F32 && !(d.epi == ub::EPI_HEAD &&
                                             (d.logits_type == ub::LOGITS_F16 || d.logits_type == ub::LOGITS_BF16)))
        return fail(UNETB200_EINVAL, "unknown logits_type");
    st->conv = pick_conv(d.taps, bn, d.amode, d.epi, d.stem_cin, d.ncls, d.pair != 0, d.stem_fmt, d.logits_type);
    if (!st->conv.fn)
        return fail(UNETB200_EINVAL, "conv: no kernel for this configuration (A_COL3 and the patch stem exist only in "
                                     "builds with -DUNETB200_TEST_VARIANTS)");
    ub::ConvParams& p = st->cp;
    memset(&p, 0, sizeof p);
    int boxW = 8, boxH = 16;
    if (d.taps == 9 && d.amode == ub::A_COL3) boxH = 18;
    if (d.taps == 9 && d.amode == ub::A_HALO) { boxW = 10; boxH = 18; }
    int rc;
    if (stem) {
        p.stem_x = d.stem_x;
        p.stem_fmt = d.stem_fmt;
        p.stem_w = d.w;
        if (stemp) {
            // tmA0/tmA1 are never used by the patch stem (it reads the input itself); keep them valid
            if ((rc = make_act_map(&p.tmA0, d.out, d.cout, d.wd, d.h, d.n, 8, 16))) return rc;
        } else if ((rc = make_input_map(&p.tmA0, d.stem_x, d.stem_fmt, d.stem_cin, d.wd, d.h, d.n))) {
            return rc;                  // im2col stem: the tile's input halo patch is one TMA box
        }
        p.tmA1 = p.tmA0;
    } else if ((rc = make_act_map(&p.tmA0, d.src0, d.c0, d.wd, d.h, d.n, boxW, boxH))) {
        return rc;
    }
    if (!stem) {
        if (d.c1 > 0) {
            if ((rc = make_act_map(&p.tmA1, d.src1, d.c1, d.wd, d.h, d.n, boxW, boxH))) return rc;
        } else {
            p.tmA1 = p.tmA0;
        }
    }
    const int cin = (stem && !stemp) ? 128 : d.c0 + d.c1;   // K extent of the packed weights (im2col stem: hi/lo layout)
    if (stemp) {
        p.tmB = p.tmA0;                 // unused: the kernel copies the weight tiles itself
    } else if ((rc = make_w_map(&p.tmB, d.w, cin, cols, d.taps == 9 ? 9 : 1, st->conv.pair ? bn / 2 : bn, st->conv.tpb))) {
        return rc;
    }
    if (d.epi == ub::EPI_UPSAMPLE) {
        const int ho = 2 * d.h, wo = 2 * d.wd;
        for (int tap = 0; tap < 4; ++tap) {
            const int a = tap >> 1, b = tap & 1;
            const char* base = static_cast<const char*>(d.out) + (uint64_t(a) * wo + b) * d.cout * 2;
            if ((rc = make_map4(&p.tmOut[tap], base, d.cout, d.wd, d.h, d.n, uint64_t(2) * d.cout * 2,
                                uint64_t(2) * wo * d.cout * 2, uint64_t(ho) * wo * d.cout * 2, 8, 4)))
                return rc;
        }
    } else if (d.epi != ub::EPI_HEAD) {
        // store boxes: one epilogue warp's quarter tile (8 x 4 pixels), pooled 4 x 2
        if ((rc = make_act_map(&p.tmOut[0], d.out, d.cout, d.wd, d.h, d.n, 8, 4))) return rc;
        for (int i = 1; i < 4; ++i) p.tmOut[i] = p.tmOut[0];
    }
    if (d.epi == ub::EPI_STORE_POOL) {
        if (!d.pool) return fail(UNETB200_EINVAL, "pool output missing");
        if ((rc = make_act_map(&p.tmPool, d.pool, d.cout, d.wd / 2, d.h / 2, d.n, 4, 2))) return rc;
    } else {
        p.tmPool = p.tmA0;
    }
    p.bias = d.bias;
    p.head_w = d.head_w;
    p.head_b = d.head_b;
    if (d.epi == ub::EPI_HEAD) {
        // the head epilogue reads bias and 1x1 weights as kernel parameters (constant bank): one small
        // synchronous read-back per plan
        if (!d.head_w || !d.head_b || d.ncls < 1 || d.ncls > ub::kMaxClasses)
            return fail(UNETB200_EINVAL, "fused head: weights missing");
        UB_CUDA(cudaMemcpy(p.bias_c, d.bias, sizeof p.bias_c, cudaMemcpyDeviceToHost));
        UB_CUDA(cudaMemcpy(p.head_wc, d.head_w, sizeof(float) * 64 * d.ncls, cudaMemcpyDeviceToHost));
        UB_CUDA(cudaMemcpy(p.head_bc, d.head_b, sizeof(float) * d.ncls, cudaMemcpyDeviceToHost));
    }
    p.logits = d.logits;
    p.mask = d.mask;
    p.mask_bits = d.mask_bits;
    p.dbg = d.dbg;
    p.C0 = d.c0;
    p.C1 = d.c1;
    p.H = d.h;
    p.W = d.wd;
    p.NIMG = d.n;
    p.Cout = d.cout;
    p.tiles_x = (d.wd + 7) / 8;
    p.tiles_y = (d.h + 15) / 16;
    p.n_blocks = cols / bn;
    const long long total = 1LL * p.tiles_x * p.tiles_y * d.n * p.n_blocks;
    if (total > 0x7fffffffLL) return fail(UNETB200_EINVAL, "conv: too many tiles");
    p.total_tiles = static_cast<int>(total);
    p.relu = d.relu;
    p.ncls = d.ncls;
    p.pf_items = d.pf_items;
    if ((rc = plan_smem(&st->conv, &p, d.taps == 9 ? 9 : 1, cin / 64, p.n_blocks, bn,
                        d.epi == ub::EPI_STORE_POOL, d.epi != ub::EPI_HEAD, stem ? 1 : d.wstat,
                        (stem && !stemp) ? ub::kStemPatchBytes : 0, d.epi2, d.min_na)))
        return rc;
    p.fd_tpi = ub::make_fastdiv(static_cast<uint32_t>(p.tiles_x * p.tiles_y));
    p.fd_tx = ub::make_fastdiv(static_cast<uint32_t>(p.tiles_x));
    p.fd_nb = ub::make_fastdiv(static_cast<uint32_t>(p.n_blocks));
    p.fd_na = ub::make_fastdiv(static_cast<uint32_t>(p.na > 0 ? p.na : 1));
    p.fd_nout = ub::make_fastdiv(static_cast<uint32_t>(p.n_out > 0 ? p.n_out : 1));
    if (st->conv.pair) {
        const long long m_tiles = 1LL * p.tiles_x * p.tiles_y * d.n;
        const long long units = (m_tiles + 1) / 2 * p.n_blocks;
        const long long pairs = units < num_sms / 2 ? units : num_sms / 2;
        st->grid = dim3(static_cast<unsigned>(2 * pairs));
    } else {
        st->grid = dim3(static_cast<unsigned>(total < num_sms ? total : num_sms));
    }
    st->block = dim3(stemp ? 512 : (stem ? 640 : 384));
    return 0;
}

int launch_step(Step& st, cudaStream_t stream) {
    if (st.kind == 1) {
        static std::mutex mu;
        static std::map<const void*, int> configured;
        {
            std::lock_guard<std::mutex> g(mu);
            int dev = 0;
            cudaGetDevice(&dev);
            auto it = configured.find(reinterpret_cast<const void*>(st.conv.fn));
            if (it == configured.end() || !(it->second & (1 << dev))) {
                UB_CUDA(cudaFuncSetAttribute(reinterpret_cast<const void*>(st.conv.fn),
                                             cudaFuncAttributeMaxDynamicSharedMemorySize,
                                             ub::kSmemLimit - ((st.conv.row || st.conv.phase) ? ub::kRowStatic : ub::kStaticSmem)));
                configured[reinterpret_cast<const void*>(st.conv.fn)] |= (1 << dev);
            }
        }
        cudaLaunchConfig_t cfg;
        memset(&cfg, 0, sizeof cfg);
        cfg.gridDim = st.grid;
        cfg.blockDim = st.block;
        cfg.dynamicSmemBytes = st.conv.smem;
        cfg.stream = stream;
        cudaLaunchAttribute attrs[2];
        int na = 0;
        if (st.conv.pair) {
            attrs[na].id = cudaLaunchAttributeClusterDimension;
            attrs[na].val.clusterDim.x = 2;
            attrs[na].val.clusterDim.y = 1;
            attrs[na].val.clusterDim.z = 1;
            ++na;
        }
        if (st.pdl) {
            attrs[na].id = cudaLaunchAttributeProgrammaticStreamSerialization;
            attrs[na].val.programmaticStreamSerializationAllowed = 1;
            ++na;
        }
        cfg.attrs = attrs;
        cfg.numAttrs = na;
        UB_CUDA(cudaLaunchKernelEx(&cfg, st.conv.fn, st.cp));
    } else {
        if (!st.stem_fn) return fail(UNETB200_EINVAL, "stem: no kernel for this configuration");
        st.stem_fn<<<st.grid, st.block, 0, stream>>>(st.sp);
    }
    UB_CUDA(cudaGetLastError());
    return 0;
}

// CUDA-core stem: fp32 NCHW and uint8 NHWC share the run-time-format instantiation; every other format has its own
template <int CIN>
StemKernel stem_cc_pick_fmt(int x_fmt) {
    switch (x_fmt) {
        case UNETB200_X_F32_NCHW:
        case UNETB200_X_U8_NHWC: return ub::stem_conv_kernel<CIN>;
        case UNETB200_X_F16_NCHW: return ub::stem_conv_kernel<CIN, ub::X_F16_NCHW>;
        case UNETB200_X_BF16_NCHW: return ub::stem_conv_kernel<CIN, ub::X_BF16_NCHW>;
        case UNETB200_X_F32_NHWC: return ub::stem_conv_kernel<CIN, ub::X_F32_NHWC>;
        case UNETB200_X_F16_NHWC: return ub::stem_conv_kernel<CIN, ub::X_F16_NHWC>;
        case UNETB200_X_BF16_NHWC: return ub::stem_conv_kernel<CIN, ub::X_BF16_NHWC>;
    }
    return nullptr;
}

int build_stem_step(const void* x, int x_fmt, int cin, const float* w, const float* bias, int n,
                    int h, int wd, void* out, Step* st) {
    if (!valid_x_fmt(x_fmt)) return fail(UNETB200_EINVAL, "unknown x_fmt");
    switch (cin) {
        case 1: st->stem_fn = stem_cc_pick_fmt<1>(x_fmt); break;
        case 3: st->stem_fn = stem_cc_pick_fmt<3>(x_fmt); break;
        case 4: st->stem_fn = stem_cc_pick_fmt<4>(x_fmt); break;
        default: return fail(UNETB200_EINVAL, "stem: n_channels must be 1, 3 or 4");
    }
    if (reinterpret_cast<uintptr_t>(x) % ub::x_elem_bytes(x_fmt))
        return fail(UNETB200_EINVAL, "stem: the input tensor is not aligned to its element size");
    st->kind = 0;
    st->stem_cin = cin;
    st->sp.x = x;
    st->sp.w = w;
    st->sp.bias = bias;
    st->sp.out = out;
    st->sp.N = n;
    st->sp.H = h;
    st->sp.W = wd;
    st->sp.x_fmt = x_fmt;
    st->grid = dim3((wd + ub::kStemTX - 1) / ub::kStemTX, (h + ub::kStemTY - 1) / ub::kStemTY, n);
    st->block = dim3(256);
    if (n > 65535) return fail(UNETB200_EINVAL, "stem: batch too large for one launch");
    return 0;
}

// First conv on the tensor cores (conv_tc.cuh, A_STEM): im2col rows built in-kernel from the
// user's tensor, hi/lo-split bf16 GEMM over two K slices against the [64][128] packed weights.
int build_stem_tc_step(const void* x, int x_fmt, int cin, const void* w_tc, const float* bias, int n,
                       int h, int wd, void* out, int num_sms, int* dbg, Step* st, bool patch = false) {
    if (!valid_x_fmt(x_fmt)) return fail(UNETB200_EINVAL, "unknown x_fmt");
    if (patch && x_fmt != UNETB200_X_F32_NCHW && x_fmt != UNETB200_X_U8_NHWC)
        return fail(UNETB200_EINVAL, "patch stem (stem_tc = 2): fp32 NCHW and uint8 NHWC inputs only; the fp16 / bf16 and "
                                     "NHWC float formats run on stem_tc = 0 or 1");
    if (patch ? !(cin == 1 || cin == 3 || cin == 4) : !(cin == 1 || cin == 3))
        return fail(UNETB200_EINVAL, "tensor-core stem: unsupported n_channels");
    ConvDesc d;
    d.c0 = 64; d.w = w_tc; d.bias = bias; d.n = n; d.h = h; d.wd = wd; d.cout = 64; d.relu = 1;
    d.taps = patch ? 9 : 1; d.epi = ub::EPI_STORE; d.out = out; d.bn = 64; d.amode = patch ? ub::A_STEMP : ub::A_STEM;
    d.stem_x = x; d.stem_fmt = x_fmt; d.stem_cin = cin; d.dbg = dbg;
    return build_conv_step(d, num_sms, st);
}

int device_num_sms(int* out) {
    int dev = 0;
    UB_CUDA(cudaGetDevice(&dev));
    UB_CUDA(cudaDeviceGetAttribute(out, cudaDevAttrMultiProcessorCount, dev));
    return 0;
}

int check_sm100() {
    int dev = 0, major = 0;
    UB_CUDA(cudaGetDevice(&dev));
    UB_CUDA(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev));
    if (major != 10)
        return fail(UNETB200_EARCH,
                    "unetb200 needs an sm_100 (B200) device; found compute capability major " +
                        std::to_string(major) + " -- there is no fallback path");
    return 0;
}

// (x, x_fmt, n, H, W, workspace, logits, logits_type, mask, mask_bits): everything baked into a plan's launches
typedef std::tuple<const void*, int, int, int, int, void*, void*, int, uint8_t*, int> PlanKey;

struct Plan {
    std::vector<Step> steps;
    // The plan's launches as ONE instantiated CUDA graph (built on the second use of a plan): a small-batch forward
    // is 22 launches of ~10-20 us each, so a host that needs more than that per cudaLaunchKernelEx starves the GPU
    // (batch-1 latency measured between 0.41 and 0.55 ms eager, depending on the host, against 0.39 ms replayed).
    cudaGraphExec_t exec = nullptr;
    float exec_thr[ub::kMaxClasses] = {};   // thresholds baked into the graph's last kernel node
    int uses = 0;
    bool graph_failed = false;
};

void destroy_plans(std::map<PlanKey, Plan>& plans) {
    for (auto& kv : plans)
        if (kv.second.exec) cudaGraphExecDestroy(kv.second.exec);
    plans.clear();
}

}  // namespace

struct unetb200_handle_s {
    unetb200_arch_t arch;
    std::vector<unetb200_layer_t> layers;
    const char* blob = nullptr;
    uint64_t blob_bytes = 0;
    int device = 0;
    int num_sms = 0;
    int amode = ub::A_HALO;
    int bn_max = 256;
    int wstat = 1;
    int stem_tc = 1;            // first conv: 0 = CUDA cores, 1 = tensor cores + in-kernel im2col (fastest measured),
                                // 2 = tensor cores, implicit GEMM over a shared-memory patch (validated, 1.6x slower)
    int pf_items = 0;           // L2 prefetch distance of the activation producer, in ring items (measured: no gain)
    int epi2 = 1;               // two epilogue groups: 0 never, 1 weight-stationary launches, 2 always
    int min_na = 3;             // weight-stationary launches: activation stages wanted before staging slots
    int pair = 2;               // CTA pairs (cta_group::2): 0 = never, 1 = wherever instantiated, 2 = where measured faster
    int pdl = 1;                // programmatic dependent launch between the layers of one forward
    int fill_sms = 1;           // narrow the column block of launches whose tiles do not cover the SMs (small batches)
    int row64 = 2;              // 64-output-channel 3x3 convs on the row-stacked kernel (conv_row.cuh): bit 0 = the
                                // one-slice layers (down1.net.3, conv1.net.3: measured equal / 5 % slower, off),
                                // bit 1 = conv1.net.0 (measured 3-5 % faster, on)
    int fold_up = 15;           // bit k: decoder level k (H >> k; bit 3 = up4 + conv4.net.0) runs as ONE launch with the
                                // up-conv folded into the 3x3 conv (conv_phase.cuh); masked by `fold_avail`
    int ps64 = 3;               // 64 -> 64 channel convs on the phase-stacked kernel (conv_ps64.cuh): bit 0 = down1.net.3,
                                // bit 1 = conv1.net.3 + head
    int fold_stack = 1;         // folded level 1 (up1 + conv1.net.0) on the phase-stacked kernel (conv_phase_stack.cuh)
    int fold_one_phase = 0;     // A/B: folded levels run one phase per work unit whatever the column block
    int fold_avail = 0;         // levels whose composite weights were packed into the blob (unetb200_pack_fused_up)
    std::vector<FusedUp> fused;
    std::vector<int> last_layers;   // layer-table row of every launch of the last forward
    int graph = 1;              // replay a plan's launches as one CUDA graph from its second use on
    cudaStream_t cap_stream = nullptr;   // capture stream of those graphs (the caller's may be the legacy stream)
    int profile = 0;
    int* dbg = nullptr;         // pinned, device-visible watchdog record
    std::map<PlanKey, Plan> plans;
    std::vector<cudaEvent_t> events;
    int last_launches = 0;
    bool timed = false;
    std::mutex mu;
};

namespace {

struct WsLayout {
    uint64_t a[5], c[4], p[4], bt, u[4], ca[4], cc[4], total;
};

// Workspace carve-up (bf16 NHWC).  Level k has (H>>k) x (W>>k) pixels and 64<<k channels.
WsLayout ws_layout(int n, int h, int w, int bw) {
    WsLayout L;
    uint64_t off = 0;
    auto take = [&](uint64_t elems) {
        uint64_t o = off;
        off = (off + elems * 2 + 1023) / 1024 * 1024;
        return o;
    };
    auto px = [&](int k) { return uint64_t(n) * (h >> k) * (w >> k); };
    for (int k = 0; k < 5; ++k) L.a[k] = take(px(k) * (uint64_t(bw) << k));        // first conv of level k
    for (int k = 0; k < 4; ++k) L.c[k] = take(px(k) * (uint64_t(bw) << k));        // skip tensors c1..c4
    for (int k = 0; k < 4; ++k) L.p[k] = take(px(k + 1) * (uint64_t(bw) << k));    // pooled p1..p4
    L.bt = take(px(4) * (uint64_t(bw) << 4));                                      // bottleneck output
    for (int k = 0; k < 4; ++k) {
        L.u[k] = L.a[k];                                   // up_k output reuses the dead a_k buffer
        L.ca[k] = take(px(k) * (uint64_t(bw) << k));       // first decoder conv of level k
        L.cc[k] = k == 0 ? 0 : take(px(k) * (uint64_t(bw) << k));   // second decoder conv (level 0: fused head)
    }
    L.total = off;
    return L;
}

int build_plan(unetb200_handle_t h, const void* x, int x_fmt, int n, int H, int W, void* ws,
               void* logits, int logits_type, uint8_t* mask, int mask_bits, Plan* plan) {
    const int bw = h->arch.base_width;
    const WsLayout L = ws_layout(n, H, W, bw);
    char* base = static_cast<char*>(ws);
    auto P = [&](uint64_t off) { return static_cast<void*>(base + off); };
    auto Wp = [&](int li) { return static_cast<const void*>(h->blob + h->layers[li].w_off); };
    auto Bp = [&](int li) { return reinterpret_cast<const float*>(h->blob + h->layers[li].b_off); };
    int rc;
    auto conv = [&](int li, const void* s0, int c0, const void* s1, int c1, int lvl, void* out,
                    void* pool) -> int {
        ConvDesc d;
        d.src0 = s0; d.c0 = c0; d.src1 = s1; d.c1 = c1;
        d.w = Wp(li); d.bias = Bp(li);
        d.n = n; d.h = H >> lvl; d.wd = W >> lvl; d.cout = h->layers[li].cout;
        d.relu = 1; d.taps = 9; d.epi = pool ? ub::EPI_STORE_POOL : ub::EPI_STORE;
        d.out = out; d.pool = pool;
        d.bn = h->bn_max; d.amode = h->amode; d.wstat = h->wstat; d.pf_items = h->pf_items; d.epi2 = h->epi2; d.min_na = h->min_na; d.dbg = h->dbg; d.fill_sms = h->fill_sms;
        if (d.cout == 64 && (h->row64 & (c1 > 0 ? 2 : 1))) d.amode = ub::A_ROW;   // bit 0: one-slice layers, bit 1: conv1.net.0
        if (d.cout == 64 && c0 == 64 && c1 == 0 && (h->ps64 & 1)) d.amode = ub::A_PS64;
        // measured on B200 (profiles/): CTA pairs win or tie on every 3x3 conv, lose slightly on the up-convs
        d.pair = h->pair >= 1;
        Step st;
        if ((rc = build_conv_step(d, h->num_sms, &st))) return rc;
        st.layer = li;
        plan->steps.push_back(st);
        return 0;
    };
    auto convt = [&](int li, const void* s, int lvl, void* out) -> int {
        ConvDesc d;
        d.src0 = s; d.c0 = h->layers[li].cin;
        d.w = Wp(li); d.bias = Bp(li);
        d.n = n; d.h = H >> lvl; d.wd = W >> lvl; d.cout = h->layers[li].cout;
        d.relu = 0; d.taps = 1; d.epi = ub::EPI_UPSAMPLE; d.out = out;
        d.bn = h->bn_max; d.amode = ub::A_TAP; d.wstat = h->wstat; d.pf_items = h->pf_items; d.epi2 = h->epi2; d.min_na = h->min_na; d.pair = h->pair == 1; d.dbg = h->dbg; d.fill_sms = h->fill_sms;
        Step st;
        if ((rc = build_conv_step(d, h->num_sms, &st))) return rc;
        st.layer = li;
        plan->steps.push_back(st);
        return 0;
    };
    // ---- encoder (unet_model.py:56-66)
    {
        Step st;
        if (h->stem_tc == 2) {
            if ((rc = build_stem_tc_step(x, x_fmt, h->arch.n_channels,
                                         h->blob + h->layers[0].w_off + stem_patch_offset(h->arch.n_channels, bw),
                                         Bp(0), n, H, W, P(L.a[0]), h->num_sms, h->dbg, &st, true)))
                return rc;
        } else if (h->stem_tc == 1 && h->arch.n_channels <= 3) {
            if ((rc = build_stem_tc_step(x, x_fmt, h->arch.n_channels,
                                         h->blob + h->layers[0].w_off + stem_tc_offset(h->arch.n_channels, bw),
                                         Bp(0), n, H, W, P(L.a[0]), h->num_sms, h->dbg, &st)))
                return rc;
        } else if ((rc = build_stem_step(x, x_fmt, h->arch.n_channels, reinterpret_cast<const float*>(Wp(0)),
                                         Bp(0), n, H, W, P(L.a[0]), &st))) {
            return rc;
        }
        st.layer = 0;
        plan->steps.push_back(st);
    }
    if ((rc = conv(1, P(L.a[0]), bw, nullptr, 0, 0, P(L.c[0]), P(L.p[0])))) return rc;
    for (int k = 1; k <= 3; ++k) {
        const int ci = bw << (k - 1), co = bw << k;
        if ((rc = conv(2 * k, P(L.p[k - 1]), ci, nullptr, 0, k, P(L.a[k]), nullptr))) return rc;
        if ((rc = conv(2 * k + 1, P(L.a[k]), co, nullptr, 0, k, P(L.c[k]), P(L.p[k])))) return rc;
    }
    // ---- bottleneck (:68)
    if ((rc = conv(8, P(L.p[3]), bw << 3, nullptr, 0, 4, P(L.a[4]), nullptr))) return rc;
    if ((rc = conv(9, P(L.a[4]), bw << 4, nullptr, 0, 4, P(L.bt), nullptr))) return rc;
    // ---- decoder (:70-84): up_k -> cat([up, skip]) -> DoubleConv
    const void* prev = P(L.bt);
    for (int k = 3; k >= 0; --k) {
        const int li_up = 10 + 3 * (3 - k);
        const int co = bw << k;
        if ((h->fold_up & h->fold_avail) >> k & 1) {
            // up_{k+1} folded into conv_{k+1}.net.0: one launch over the low-resolution tensor and the skip tensor
            const FusedUp& f = h->fused[k + 1];
            PhaseDesc d;
            d.low = prev; d.c_low = f.clow; d.skip = P(L.c[k]); d.c_skip = co;
            d.wc = h->blob + f.w_off; d.w3 = Wp(li_up + 1); d.c_up = f.cmid;
            d.bias9 = reinterpret_cast<const float*>(h->blob + f.b_off);
            d.n = n; d.h = H >> (k + 1); d.wd = W >> (k + 1); d.cout = f.cout; d.relu = 1;
            d.out = P(L.ca[k]); d.bn = h->bn_max; d.pair = h->pair >= 1; d.dbg = h->dbg;
            d.one_phase = h->fold_one_phase; d.stack = h->fold_stack; d.fill_sms = h->fill_sms;
            Step st;
            if ((rc = build_phase_step(d, h->num_sms, &st))) return rc;
            st.layer = li_up + 1;
            plan->steps.push_back(st);
        } else {
            if ((rc = convt(li_up, prev, k + 1, P(L.u[k])))) return rc;
            if ((rc = conv(li_up + 1, P(L.u[k]), co, P(L.c[k]), co, k, P(L.ca[k]), nullptr))) return rc;
        }
        if (k > 0) {
            if ((rc = conv(li_up + 2, P(L.ca[k]), co, nullptr, 0, k, P(L.cc[k]), nullptr))) return rc;
            prev = P(L.cc[k]);
        } else {
            // conv1.net.3 + out_conv (:86) + threshold (inference.py:72-79) in one kernel
            ConvDesc d;
            d.src0 = P(L.ca[0]); d.c0 = bw;
            d.w = Wp(21); d.bias = Bp(21);
            d.n = n; d.h = H; d.wd = W; d.cout = bw; d.relu = 1; d.taps = 9; d.epi = ub::EPI_HEAD;
            d.head_w = reinterpret_cast<const float*>(Wp(22)); d.head_b = Bp(22);
            d.ncls = h->arch.n_classes; d.logits = logits; d.logits_type = logits_type; d.mask = mask; d.mask_bits = mask_bits;
            d.bn = 64; d.amode = (h->ps64 & 2) ? ub::A_PS64 : ((h->row64 & 1) ? ub::A_ROW : h->amode); d.wstat = h->wstat; d.pf_items = h->pf_items; d.epi2 = h->epi2; d.min_na = h->min_na; d.pair = h->pair >= 1; d.dbg = h->dbg;
            Step st;
            if ((rc = build_conv_step(d, h->num_sms, &st))) return rc;
            st.layer = 21;
            plan->steps.push_back(st);
        }
    }
    return 0;
}

}  // namespace

// ====================================================================== C ABI
extern "C" {

int unetb200_abi_version(void) { return UNETB200_ABI_VERSION; }
int unetb200_build_flags(void) {
#ifdef UNETB200_TEST_VARIANTS
    return UNETB200_BUILD_TEST_VARIANTS;
#else
    return 0;
#endif
}
const char* unetb200_last_error(void) { return g_err.c_str(); }

int unetb200_num_layers(const unetb200_arch_t* arch) {
    if (check_arch(arch)) return -1;
    return static_cast<int>(layer_table(*arch).size());
}

int unetb200_layer_info(const unetb200_arch_t* arch, int index, unetb200_layer_t* out) {
    int rc = check_arch(arch);
    if (rc) return rc;
    if (!out) return fail(UNETB200_EINVAL, "out is NULL");
    auto t = layer_table(*arch);
    if (index < 0 || index >= static_cast<int>(t.size())) return fail(UNETB200_EINVAL, "layer index out of range");
    *out = t[index];
    return 0;
}

uint64_t unetb200_packed_bytes(const unetb200_arch_t* arch) {
    if (check_arch(arch)) return 0;
    return fused_table(*arch)[0].w_off;      // per-layer regions, then the folded up-conv levels
}

int unetb200_fused_up_info(const unetb200_arch_t* arch, int level, uint64_t* w_off, uint64_t* w_bytes,
                           uint64_t* b_off, uint64_t* b_bytes) {
    int rc = check_arch(arch);
    if (rc) return rc;
    if (level < 1 || level > 4) return fail(UNETB200_EINVAL, "fused up-conv level must be 1..4");
    const FusedUp f = fused_table(*arch)[level];
    if (w_off) *w_off = f.w_off;
    if (w_bytes) *w_bytes = f.w_bytes;
    if (b_off) *b_off = f.b_off;
    if (b_bytes) *b_bytes = f.b_bytes;
    return 0;
}

int unetb200_pack_fused_up(const unetb200_arch_t* arch, int level, const float* up_weight, const float* up_bias,
                           const float* conv_weight, const float* conv_bias, const float* bn_gamma,
                           const float* bn_beta, const float* bn_mean, const float* bn_var, float bn_eps,
                           void* blob_dev, void* stream) {
    int rc = check_arch(arch);
    if (rc) return rc;
    if (level < 1 || level > 4) return fail(UNETB200_EINVAL, "fused up-conv level must be 1..4");
    if (!up_weight || !conv_weight || !blob_dev) return fail(UNETB200_EINVAL, "weight/blob pointer is NULL");
    if (bn_gamma && (!bn_beta || !bn_mean || !bn_var))
        return fail(UNETB200_EINVAL, "BatchNorm needs gamma, beta, mean and var together");
    const FusedUp f = fused_table(*arch)[level];
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    char* blob = static_cast<char*>(blob_dev);
    const int cin3 = 2 * f.cmid;                 // conv{level}.net.0 reads cat([up, skip])
    ub::pack_fused_up_w_kernel<<<dim3(f.clow / 64, f.cout / 64, 16), 256, 0, s>>>(
        up_weight, conv_weight, bn_gamma, bn_var, bn_eps, f.clow, f.cmid, cin3, f.cout,
        reinterpret_cast<uint16_t*>(blob + f.w_off));
    ub::pack_fused_up_b_kernel<<<(9 * f.cout + 127) / 128, 128, 0, s>>>(
        up_bias, conv_weight, conv_bias, bn_gamma, bn_beta, bn_mean, bn_var, bn_eps, f.cmid, cin3, f.cout,
        reinterpret_cast<float*>(blob + f.b_off), reinterpret_cast<uint32_t*>(blob + f.flag_off));
    UB_CUDA(cudaGetLastError());
    return 0;
}

int unetb200_pack_layer(const unetb200_arch_t* arch, int index, const float* weight,
                        const float* bias, const float* bn_gamma, const float* bn_beta,
                        const float* bn_mean, const float* bn_var, float bn_eps, void* blob_dev,
                        void* stream) {
    int rc = check_arch(arch);
    if (rc) return rc;
    auto t = layer_table(*arch);
    if (index < 0 || index >= static_cast<int>(t.size())) return fail(UNETB200_EINVAL, "layer index out of range");
    if (!weight || !blob_dev) return fail(UNETB200_EINVAL, "weight/blob pointer is NULL");
    if (bn_gamma && (!bn_beta || !bn_mean || !bn_var))
        return fail(UNETB200_EINVAL, "BatchNorm needs gamma, beta, mean and var together");
    const unetb200_layer_t& l = t[index];
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    char* blob = static_cast<char*>(blob_dev);
    float* db = reinterpret_cast<float*>(blob + l.b_off);
    const int threads = 256;
    switch (l.kind) {
        case UNETB200_STEM: {
            const int total = 9 * l.cin * l.cout;
            ub::pack_stem_kernel<<<(total + threads - 1) / threads, threads, 0, s>>>(
                weight, bias, bn_gamma, bn_beta, bn_mean, bn_var, bn_eps, l.cout, l.cin,
                reinterpret_cast<float*>(blob + l.w_off), db);
            ub::pack_stem_tc_kernel<<<(l.cout * 128 + threads - 1) / threads, threads, 0, s>>>(
                weight, bias, bn_gamma, bn_beta, bn_mean, bn_var, bn_eps, l.cout, l.cin,
                reinterpret_cast<uint16_t*>(blob + l.w_off + stem_tc_offset(l.cin, l.cout)));
            ub::pack_stem_patch_kernel<<<(9 * 32 * l.cout + threads - 1) / threads, threads, 0, s>>>(   // 9 x 2 x cout x 16
                weight, bn_gamma, bn_var, bn_eps, l.cout, l.cin,
                reinterpret_cast<uint16_t*>(blob + l.w_off + stem_patch_offset(l.cin, l.cout)));
            break;
        }
        case UNETB200_CONV3X3: {
            const uint64_t total = uint64_t(9) * l.cin * l.cout;
            uint64_t blocks = (total + threads - 1) / threads;
            if (blocks > 65535 * 4) blocks = 65535 * 4;
            ub::pack_conv3x3_kernel<<<static_cast<unsigned>(blocks), threads, 0, s>>>(
                weight, bias, bn_gamma, bn_beta, bn_mean, bn_var, bn_eps, l.cout, l.cin,
                reinterpret_cast<uint16_t*>(blob + l.w_off), db);
            break;
        }
        case UNETB200_CONVT2X2: {
            const uint64_t total = uint64_t(4) * l.cin * l.cout;
            uint64_t blocks = (total + threads - 1) / threads;
            ub::pack_convt_kernel<<<static_cast<unsigned>(blocks), threads, 0, s>>>(
                weight, bias, l.cin, l.cout, reinterpret_cast<uint16_t*>(blob + l.w_off), db);
            break;
        }
        case UNETB200_HEAD: {
            // Conv2d 1x1 weight [ncls][64][1][1] is already [ncls][64]
            UB_CUDA(cudaMemcpyAsync(blob + l.w_off, weight, l.w_bytes, cudaMemcpyDeviceToDevice, s));
            if (bias)
                UB_CUDA(cudaMemcpyAsync(db, bias, l.b_bytes, cudaMemcpyDeviceToDevice, s));
            else
                UB_CUDA(cudaMemsetAsync(db, 0, l.b_bytes, s));
            break;
        }
    }
    UB_CUDA(cudaGetLastError());
    return 0;
}

int unetb200_create(const unetb200_arch_t* arch, const void* blob_dev, uint64_t blob_bytes,
                    int device, unetb200_handle_t* out) {
    int rc = check_arch(arch);
    if (rc) return rc;
    if (!blob_dev || !out) return fail(UNETB200_EINVAL, "blob/out pointer is NULL");
    const std::vector<FusedUp> fused = fused_table(*arch);
    // the folded up-conv regions are optional: a blob that ends after the per-layer regions runs the unfused plan
    const bool has_fused = blob_bytes >= fused[0].w_off;
    if (blob_bytes < fused[4].w_off) return fail(UNETB200_EINVAL, "weights blob too small");
    UB_CUDA(cudaSetDevice(device));
    if ((rc = check_sm100())) return rc;
    if (!encode_tiled()) return fail(UNETB200_ECUDA, "cuTensorMapEncodeTiled entry point unavailable");
    unetb200_handle_t h = new unetb200_handle_s();
    h->arch = *arch;
    h->layers = layer_table(*arch);
    h->blob = static_cast<const char*>(blob_dev);
    h->blob_bytes = blob_bytes;
    h->device = device;
    if ((rc = device_num_sms(&h->num_sms))) { delete h; return rc; }
    cudaError_t e = cudaHostAlloc(reinterpret_cast<void**>(&h->dbg), 64, cudaHostAllocMapped);
    if (e != cudaSuccess) { delete h; return fail(UNETB200_ECUDA, "cudaHostAlloc(dbg) failed"); }
    memset(h->dbg, 0, 64);
    h->fused = fused;
    if (has_fused) {
        for (int j = 1; j <= 4; ++j) {
            uint32_t flag = 0;
            if (cudaMemcpy(&flag, h->blob + fused[j].flag_off, 4, cudaMemcpyDeviceToHost) != cudaSuccess) {
                cudaFreeHost(h->dbg);
                delete h;
                return fail(UNETB200_ECUDA, "reading the blob failed");
            }
            if (flag == 0x46555345u) h->fold_avail |= 1 << (j - 1);
        }
    }
    const char* env = getenv("UNETB200_FOLD_UP");
    if (env) h->fold_up = atoi(env) & 15;
    env = getenv("UNETB200_PS64");
    if (env) h->ps64 = atoi(env) & 3;
    env = getenv("UNETB200_FOLD_STACK");
    if (env) h->fold_stack = atoi(env) ? 1 : 0;
    env = getenv("UNETB200_FOLD_ONE_PHASE");
    if (env) h->fold_one_phase = atoi(env) ? 1 : 0;
    env = getenv("UNETB200_AMODE");
    if (env) h->amode = atoi(env);
    env = getenv("UNETB200_BN_MAX");
    if (env) h->bn_max = atoi(env);
    env = getenv("UNETB200_WSTAT");
    if (env) h->wstat = atoi(env) ? 1 : 0;
    env = getenv("UNETB200_PDL");
    if (env) h->pdl = atoi(env) ? 1 : 0;
    env = getenv("UNETB200_PAIR");
    if (env) h->pair = atoi(env);
    env = getenv("UNETB200_EPI2");
    if (env) h->epi2 = atoi(env);
    env = getenv("UNETB200_PF_ITEMS");
    if (env) h->pf_items = atoi(env);
    env = getenv("UNETB200_STEM_TC");
    if (env) h->stem_tc = atoi(env);
    env = getenv("UNETB200_ROW64");
    if (env) h->row64 = atoi(env) & 3;
    *out = h;
    return 0;
}

int unetb200_destroy(unetb200_handle_t h) {
    if (!h) return 0;
    for (cudaEvent_t e : h->events) cudaEventDestroy(e);
    destroy_plans(h->plans);
    if (h->cap_stream) cudaStreamDestroy(h->cap_stream);
    if (h->dbg) cudaFreeHost(h->dbg);
    delete h;
    return 0;
}

int unetb200_set_option(unetb200_handle_t h, const char* key, int value) {
    if (!h || !key) return fail(UNETB200_EINVAL, "handle/key is NULL");
    std::lock_guard<std::mutex> g(h->mu);
    std::string k(key);
    if (k == "amode") {
        if (value < 0 || value > 2) return fail(UNETB200_EINVAL, "amode must be 0..2");
        h->amode = value;
    } else if (k == "bn_max") {
        if (!(value == 64 || value == 128 || value == 256)) return fail(UNETB200_EINVAL, "bn_max must be 64/128/256");
        h->bn_max = value;
    } else if (k == "wstat") {
        h->wstat = value ? 1 : 0;
    } else if (k == "stem_tc") {
        if (value < 0 || value > 2) return fail(UNETB200_EINVAL, "stem_tc must be 0, 1 or 2");
        h->stem_tc = value;
    } else if (k == "pdl") {
        h->pdl = value ? 1 : 0;
    } else if (k == "pair") {
        if (value < 0 || value > 2) return fail(UNETB200_EINVAL, "pair must be 0, 1 or 2");
        h->pair = value;
    } else if (k == "min_na") {
        if (value < 2 || value > 8) return fail(UNETB200_EINVAL, "min_na must be in 2..8");
        h->min_na = value;
    } else if (k == "epi2") {
        if (value < 0 || value > 2) return fail(UNETB200_EINVAL, "epi2 must be 0, 1 or 2");
        h->epi2 = value;
    } else if (k == "pf_items") {
        if (value < 0 || value > 64) return fail(UNETB200_EINVAL, "pf_items must be in 0..64");
        h->pf_items = value;
    } else if (k == "fill_sms") {
        if (value < 0 || value > 2) return fail(UNETB200_EINVAL, "fill_sms must be 0, 1 or 2");
        h->fill_sms = value;                 // 2 = also the up-convs (measured: no gain at batch 1-4)
    } else if (k == "row64") {
        if (value < 0 || value > 3) return fail(UNETB200_EINVAL, "row64 must be 0..3 (bit 0: Cin = 64 layers, bit 1: conv1.net.0)");
        h->row64 = value;
    } else if (k == "fold_up") {
        if (value < 0 || value > 15) return fail(UNETB200_EINVAL, "fold_up must be 0..15 (bit k: decoder level k)");
        h->fold_up = value;
    } else if (k == "ps64") {
        if (value < 0 || value > 3) return fail(UNETB200_EINVAL, "ps64 must be 0..3 (bit 0: down1.net.3, bit 1: conv1.net.3)");
        h->ps64 = value;
    } else if (k == "fold_one_phase") {
        h->fold_one_phase = value ? 1 : 0;
    } else if (k == "fold_stack") {
        h->fold_stack = value ? 1 : 0;
    } else if (k == "graph") {
        h->graph = value ? 1 : 0;
    } else if (k == "profile") {
        h->profile = value ? 1 : 0;
    } else {
        return fail(UNETB200_EINVAL, "unknown option " + k);
    }
    destroy_plans(h->plans);
    return 0;
}

int unetb200_get_option(unetb200_handle_t h, const char* key, int* value) {
    if (!h || !key || !value) return fail(UNETB200_EINVAL, "handle/key/value is NULL");
    std::string k(key);
    if (k == "amode") *value = h->amode;
    else if (k == "bn_max") *value = h->bn_max;
    else if (k == "wstat") *value = h->wstat;
    else if (k == "stem_tc") *value = h->stem_tc;
    else if (k == "pf_items") *value = h->pf_items;
    else if (k == "epi2") *value = h->epi2;
    else if (k == "min_na") *value = h->min_na;
    else if (k == "pair") *value = h->pair;
    else if (k == "pdl") *value = h->pdl;
    else if (k == "fill_sms") *value = h->fill_sms;
    else if (k == "row64") *value = h->row64;
    else if (k == "fold_up") *value = h->fold_up & h->fold_avail;
    else if (k == "fold_avail") *value = h->fold_avail;
    else if (k == "fold_one_phase") *value = h->fold_one_phase;
    else if (k == "fold_stack") *value = h->fold_stack;
    else if (k == "ps64") *value = h->ps64;
    else if (k == "graph") *value = h->graph;
    else if (k == "profile") *value = h->profile;
    else if (k == "num_sms") *value = h->num_sms;
    else return fail(UNETB200_EINVAL, "unknown option " + k);
    return 0;
}

uint64_t unetb200_workspace_bytes(unetb200_handle_t h, int n, int height, int width) {
    if (!h || n <= 0 || height <= 0 || width <= 0 || height % 16 || width % 16) return 0;
    return ws_layout(n, height, width, h->arch.base_width).total;
}

static int forward_impl(unetb200_handle_t h, const void* x, int x_fmt, int n, int height, int width,
                        void* workspace, uint64_t workspace_bytes, void* logits, int logits_type, uint8_t* mask,
                        int mask_bits, const float* logit_thr, void* stream) {
    if (!h) return fail(UNETB200_EINVAL, "handle is NULL");
    if (!x || !workspace) return fail(UNETB200_EINVAL, "x/workspace pointer is NULL");
    if (n <= 0 || height <= 0 || width <= 0) return fail(UNETB200_EINVAL, "empty input");
    if (height % 16 || width % 16)
        return fail(UNETB200_EINVAL,
                    "H and W must be divisible by 16 (the reference fails in torch.cat otherwise), got " +
                        std::to_string(height) + "x" + std::to_string(width));
    if (!logits && !mask) return fail(UNETB200_EINVAL, "both outputs are NULL");
    if (!valid_x_fmt(x_fmt)) return fail(UNETB200_EINVAL, "unknown x_fmt");
    if (!(logits_type == UNETB200_LOGITS_F32 || logits_type == UNETB200_LOGITS_F16 || logits_type == UNETB200_LOGITS_BF16))
        return fail(UNETB200_EINVAL, "unknown logits_type");
    if (mask && !logit_thr) return fail(UNETB200_EINVAL, "mask requested without thresholds");
    const uint64_t need = ws_layout(n, height, width, h->arch.base_width).total;
    if (workspace_bytes < need)
        return fail(UNETB200_ENOMEM, "workspace too small: need " + std::to_string(need) + " bytes");
    if (reinterpret_cast<uintptr_t>(workspace) % 1024)
        return fail(UNETB200_EINVAL, "workspace must be 1024-byte aligned");
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    std::lock_guard<std::mutex> g(h->mu);
    if (h->dbg && h->dbg[0] == 0xDEAD) {
        // a kernel of an earlier forward ran into the bounded mbarrier wait (ptx.cuh) and trapped: the CUDA
        // context is gone; say where instead of failing with a bare "unspecified launch failure"
        char buf[200];
        snprintf(buf, sizeof buf, "an earlier launch trapped in its mbarrier watchdog (wait site %d, block %d, "
                 "thread %d, parity %d): the CUDA context of this process is unusable",
                 h->dbg[1], h->dbg[2], h->dbg[3], h->dbg[4]);
        return fail(UNETB200_ECUDA, buf);
    }
    // run on the handle's device and hand the caller's current device back on every exit path
    struct DeviceGuard {
        int prev = -1;
        bool switched = false;
        ~DeviceGuard() { if (switched) cudaSetDevice(prev); }
    } guard;
    UB_CUDA(cudaGetDevice(&guard.prev));
    if (guard.prev != h->device) {
        UB_CUDA(cudaSetDevice(h->device));
        guard.switched = true;
    }
    PlanKey key(x, x_fmt, n, height, width, workspace, logits, logits_type, mask, mask_bits);
    auto it = h->plans.find(key);
    if (it == h->plans.end()) {
        Plan plan;
        int rc = build_plan(h, x, x_fmt, n, height, width, workspace, logits, logits_type, mask, mask_bits, &plan);
        if (rc) return rc;
        if (h->plans.size() > 64) destroy_plans(h->plans);
        it = h->plans.emplace(key, std::move(plan)).first;
    }
    Plan& plan = it->second;
    if (mask) {
        Step& last = plan.steps.back();
        for (int c = 0; c < h->arch.n_classes; ++c) last.cp.thr[c] = logit_thr[c];
    }
    const bool prof = h->profile != 0;
    if (prof) {
        while (h->events.size() < plan.steps.size() + 1) {
            cudaEvent_t e;
            UB_CUDA(cudaEventCreate(&e));
            h->events.push_back(e);
        }
        UB_CUDA(cudaEventRecord(h->events[0], s));
    }
    auto launch_all = [&](cudaStream_t on) -> int {
        for (size_t i = 0; i < plan.steps.size(); ++i) {
            // the first launch of a forward keeps normal stream order (its predecessor is foreign work)
            plan.steps[i].pdl = (h->pdl && !prof && i > 0 && plan.steps[i].kind == 1) ? 1 : 0;
            int rc = launch_step(plan.steps[i], on);
            if (rc) return rc;
            if (prof) UB_CUDA(cudaEventRecord(h->events[i + 1], on));
        }
        return 0;
    };
    h->last_launches = static_cast<int>(plan.steps.size());
    h->last_layers.resize(plan.steps.size());
    for (size_t i = 0; i < plan.steps.size(); ++i) h->last_layers[i] = plan.steps[i].layer;
    h->timed = prof;
    ++plan.uses;
    // graph replay: not while profiling, not inside somebody else's capture, from the second use of a plan on
    cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
    if (h->graph && !prof && !plan.graph_failed && plan.uses >= 2 &&
        cudaStreamIsCapturing(s, &cap) == cudaSuccess && cap == cudaStreamCaptureStatusNone) {
        const int ncls = h->arch.n_classes;
        if (plan.exec && mask && memcmp(plan.exec_thr, plan.steps.back().cp.thr, sizeof(float) * ncls) != 0) {
            cudaGraphExecDestroy(plan.exec);            // other thresholds: re-capture (they are kernel parameters)
            plan.exec = nullptr;
        }
        if (!plan.exec) {
            if (!h->cap_stream && cudaStreamCreateWithFlags(&h->cap_stream, cudaStreamNonBlocking) != cudaSuccess)
                h->cap_stream = nullptr;
            cudaGraph_t g = nullptr;
            bool ok = h->cap_stream &&
                      cudaStreamBeginCapture(h->cap_stream, cudaStreamCaptureModeThreadLocal) == cudaSuccess;
            if (ok) {
                const int rc = launch_all(h->cap_stream);
                ok = cudaStreamEndCapture(h->cap_stream, &g) == cudaSuccess && rc == 0 && g != nullptr;
            }
            if (ok) ok = cudaGraphInstantiate(&plan.exec, g, 0) == cudaSuccess;
            if (g) cudaGraphDestroy(g);
            if (!ok) {
                cudaGetLastError();                     // capture problems are not sticky: fall back to direct launches
                plan.exec = nullptr;
                plan.graph_failed = true;
            } else {
                memcpy(plan.exec_thr, plan.steps.back().cp.thr, sizeof plan.exec_thr);
            }
        }
        if (plan.exec) {
            UB_CUDA(cudaGraphLaunch(plan.exec, s));
            return 0;
        }
    }
    return launch_all(s);
}

int unetb200_forward(unetb200_handle_t h, const void* x, int x_fmt, int n, int height, int width,
                     void* workspace, uint64_t workspace_bytes, float* logits, uint8_t* mask,
                     const float* logit_thr, void* stream) {
    return forward_impl(h, x, x_fmt, n, height, width, workspace, workspace_bytes, logits, UNETB200_LOGITS_F32, mask, 0,
                        logit_thr, stream);
}

int unetb200_forward_bits(unetb200_handle_t h, const void* x, int x_fmt, int n, int height, int width,
                          void* workspace, uint64_t workspace_bytes, float* logits, uint8_t* mask_bits,
                          const float* logit_thr, void* stream) {
    return forward_impl(h, x, x_fmt, n, height, width, workspace, workspace_bytes, logits, UNETB200_LOGITS_F32,
                        mask_bits, 1, logit_thr, stream);
}

int unetb200_forward_typed(unetb200_handle_t h, const void* x, int x_fmt, int n, int height, int width,
                           void* workspace, uint64_t workspace_bytes, void* logits, int logits_type,
                           uint8_t* mask, int mask_bits, const float* logit_thr, void* stream) {
    return forward_impl(h, x, x_fmt, n, height, width, workspace, workspace_bytes, logits, logits_type, mask,
                        mask_bits ? 1 : 0, logit_thr, stream);
}

int unetb200_layer_times(unetb200_handle_t h, float* ms, int count) {
    if (!h || !ms) return fail(UNETB200_EINVAL, "handle/ms is NULL");
    std::lock_guard<std::mutex> g(h->mu);
    if (!h->timed) return fail(UNETB200_EINVAL, "last forward was not profiled (set option profile=1)");
    const int nl = static_cast<int>(h->layers.size());
    for (int i = 0; i < count; ++i) ms[i] = 0.f;
    // steps follow the layer table except out_conv, which is fused into conv1.net.3
    const int nsteps = h->last_launches;
    UB_CUDA(cudaEventSynchronize(h->events[nsteps]));
    for (int i = 0; i < nsteps; ++i) {
        float t = 0.f;
        UB_CUDA(cudaEventElapsedTime(&t, h->events[i], h->events[i + 1]));
        const int li = h->last_layers[i];       // (a folded up-conv leaves its row at 0 and adds to its conv's)
        if (li >= 0 && li < count && li < nl) ms[li] += t;
    }
    return 0;
}

int unetb200_last_launch_count(unetb200_handle_t h) { return h ? h->last_launches : -1; }

// ------------------------------------------------------------------ single-kernel hooks
static int* g_hook_dbg() {
    static int* dbg = nullptr;
    if (!dbg) {
        if (cudaHostAlloc(reinterpret_cast<void**>(&dbg), 64, cudaHostAllocMapped) != cudaSuccess)
            dbg = nullptr;
        else
            memset(dbg, 0, 64);
    }
    return dbg;
}

int unetb200_conv3x3(const void* src0, int c0, const void* src1, int c1, const void* w_packed,
                     const float* bias, int n, int height, int width, int cout, int relu, void* out,
                     void* pool_out, int bn, int amode, int wstat, void* stream) {
    int rc;
    if ((rc = check_sm100())) return rc;
    if (!src0 || !w_packed || !bias || !out) return fail(UNETB200_EINVAL, "NULL pointer");
    if (pool_out && (height % 2 || width % 2)) return fail(UNETB200_EINVAL, "pool needs even H, W");
    ConvDesc d;
    d.src0 = src0; d.c0 = c0; d.src1 = src1; d.c1 = src1 ? c1 : 0;
    d.w = w_packed; d.bias = bias; d.n = n; d.h = height; d.wd = width; d.cout = cout; d.relu = relu;
    d.taps = 9; d.epi = pool_out ? ub::EPI_STORE_POOL : ub::EPI_STORE; d.out = out; d.pool = pool_out;
    d.bn = bn; d.amode = amode; d.wstat = wstat & 1; d.pair = (wstat >> 1) & 1; d.dbg = g_hook_dbg();
    int sms = 0;
    if ((rc = device_num_sms(&sms))) return rc;
    Step st;
    if ((rc = build_conv_step(d, sms, &st))) return rc;
    return launch_step(st, static_cast<cudaStream_t>(stream));
}

int unetb200_conv3x3_head(const void* src0, int c0, const void* w_packed, const float* bias,
                          const float* head_w, const float* head_b, int n_classes, int n, int height,
                          int width, void* logits, uint8_t* mask, const float* logit_thr, int amode,
                          int wstat, void* stream) {
    int rc;
    if ((rc = check_sm100())) return rc;
    const int logits_type = (wstat >> 3) & 3;
    if (logits_type == 3) return fail(UNETB200_EINVAL, "unknown logits_type (wstat bits 3-4)");
    if (!src0 || !w_packed || !bias || !head_w || !head_b) return fail(UNETB200_EINVAL, "NULL pointer");
    if (n_classes < 1 || n_classes > ub::kMaxClasses) return fail(UNETB200_EINVAL, "n_classes must be in 1..8");
    if (mask && !logit_thr) return fail(UNETB200_EINVAL, "mask requested without thresholds");
    ConvDesc d;
    d.src0 = src0; d.c0 = c0; d.w = w_packed; d.bias = bias; d.n = n; d.h = height; d.wd = width;
    d.cout = 64; d.relu = 1; d.taps = 9; d.epi = ub::EPI_HEAD; d.head_w = head_w; d.head_b = head_b;
    d.ncls = n_classes; d.logits = logits; d.mask = mask; d.bn = 64; d.amode = amode;
    d.wstat = wstat & 1; d.pair = (wstat >> 1) & 1; d.mask_bits = (wstat >> 2) & 1; d.logits_type = logits_type;
    d.dbg = g_hook_dbg();
    int sms = 0;
    if ((rc = device_num_sms(&sms))) return rc;
    Step st;
    if ((rc = build_conv_step(d, sms, &st))) return rc;
    if (mask) for (int c = 0; c < n_classes; ++c) st.cp.thr[c] = logit_thr[c];
    return launch_step(st, static_cast<cudaStream_t>(stream));
}

int unetb200_convt2x2(const void* src, int cin, const void* w_packed, const float* bias, int n,
                      int height, int width, int cout, void* out, int bn, void* stream) {
    int rc;
    if ((rc = check_sm100())) return rc;
    if (!src || !w_packed || !bias || !out) return fail(UNETB200_EINVAL, "NULL pointer");
    ConvDesc d;
    d.src0 = src; d.c0 = cin; d.w = w_packed; d.bias = bias; d.n = n; d.h = height; d.wd = width;
    d.cout = cout; d.relu = 0; d.taps = 1; d.epi = ub::EPI_UPSAMPLE; d.out = out; d.bn = bn & 0xfff;
    d.pair = (bn >> 12) & 1;     // bit 12 of `bn` selects the CTA-pair variant
    d.amode = ub::A_TAP; d.dbg = g_hook_dbg();
    int sms = 0;
    if ((rc = device_num_sms(&sms))) return rc;
    Step st;
    if ((rc = build_conv_step(d, sms, &st))) return rc;
    return launch_step(st, static_cast<cudaStream_t>(stream));
}

int unetb200_upconv3x3(const void* low, int c_low, const void* skip, int c_skip, const void* wc_packed,
                       const void* w3_packed, int c_up, const float* bias9, int n, int h_low, int w_low, int cout,
                       int relu, void* out, int bn, int flags, void* stream) {
    int rc;
    if ((rc = check_sm100())) return rc;
    if (!low || !skip || !wc_packed || !w3_packed || !bias9 || !out) return fail(UNETB200_EINVAL, "NULL pointer");
    PhaseDesc d;
    d.low = low; d.c_low = c_low; d.skip = skip; d.c_skip = c_skip; d.wc = wc_packed; d.w3 = w3_packed;
    d.c_up = c_up; d.bias9 = bias9; d.n = n; d.h = h_low; d.wd = w_low; d.cout = cout; d.relu = relu; d.out = out;
    d.bn = bn; d.pair = flags & 1; d.one_phase = (flags >> 1) & 1; d.stack = (flags >> 2) & 1; d.dbg = g_hook_dbg();
    int sms = 0;
    if ((rc = device_num_sms(&sms))) return rc;
    Step st;
    if ((rc = build_phase_step(d, sms, &st))) return rc;
    return launch_step(st, static_cast<cudaStream_t>(stream));
}

uint64_t unetb200_stem_tc_offset(int cin) { return stem_tc_offset(cin, 64); }

int unetb200_stem_tc(const void* x, int x_fmt, int cin, const void* w_tc, const float* bias, int n,
                     int height, int width, void* out, void* stream) {
    int rc;
    if ((rc = check_sm100())) return rc;
    if (!x || !w_tc || !bias || !out) return fail(UNETB200_EINVAL, "NULL pointer");
    int sms = 0;
    if ((rc = device_num_sms(&sms))) return rc;
    Step st;
    if ((rc = build_stem_tc_step(x, x_fmt, cin, w_tc, bias, n, height, width, out, sms, g_hook_dbg(), &st)))
        return rc;
    return launch_step(st, static_cast<cudaStream_t>(stream));
}

uint64_t unetb200_stem_patch_offset(int cin) { return stem_patch_offset(cin, 64); }

int unetb200_stem_patch(const void* x, int x_fmt, int cin, const void* w_patch, const float* bias, int n,
                        int height, int width, void* out, void* stream) {
    int rc;
    if ((rc = check_sm100())) return rc;
    if (!x || !w_patch || !bias || !out) return fail(UNETB200_EINVAL, "NULL pointer");
    int sms = 0;
    if ((rc = device_num_sms(&sms))) return rc;
    Step st;
    if ((rc = build_stem_tc_step(x, x_fmt, cin, w_patch, bias, n, height, width, out, sms, g_hook_dbg(), &st, true)))
        return rc;
    return launch_step(st, static_cast<cudaStream_t>(stream));
}

int unetb200_stem(const void* x, int x_fmt, int cin, const float* w, const float* bias, int n,
                  int height, int width, void* out, void* stream) {
    if (!x || !w || !bias || !out) return fail(UNETB200_EINVAL, "NULL pointer");
    Step st;
    int rc = build_stem_step(x, x_fmt, cin, w, bias, n, height, width, out, &st);
    if (rc) return rc;
    return launch_step(st, static_cast<cudaStream_t>(stream));
}

// ------------------------------------------------------------------ pre / post processing
namespace {
// Pillow's bicubic kernel (Resample.c bicubic_filter, a = -0.5), evaluated exactly as written there.
inline double pil_bicubic(double x) {
    const double a = -0.5;
    if (x < 0.0) x = -x;
    if (x < 1.0) return ((a + 2.0) * x - (a + 3.0)) * x * x + 1;
    if (x < 2.0) return (((x - 5) * x + 8) * x - 4) * a;
    return 0.0;
}
inline int pil_ksize(int in_size, int out_size) {
    double filterscale = static_cast<double>(in_size) / out_size;
    if (filterscale < 1.0) filterscale = 1.0;
    return static_cast<int>(std::ceil(2.0 * filterscale)) * 2 + 1;
}
}  // namespace

int unetb200_resize_ksize(int in_size, int out_size) {
    if (in_size <= 0 || out_size <= 0) return -1;
    return pil_ksize(in_size, out_size);
}

// precompute_coeffs + normalize_coeffs_8bpc of Pillow's Resample.c for box = (0, in_size)
int unetb200_resize_coeffs(int in_size, int out_size, int32_t* kk, int32_t* bounds) {
    if (in_size <= 0 || out_size <= 0 || !kk || !bounds) return fail(UNETB200_EINVAL, "resize_coeffs: bad argument");
    const double in0 = 0.0, in1 = static_cast<double>(in_size);
    const double scale = (in1 - in0) / out_size;
    double filterscale = scale;
    if (filterscale < 1.0) filterscale = 1.0;
    const double support = 2.0 * filterscale;
    const int ksize = static_cast<int>(std::ceil(support)) * 2 + 1;
    std::vector<double> k(ksize);
    for (int xx = 0; xx < out_size; ++xx) {
        const double center = in0 + (xx + 0.5) * scale;
        double ww = 0.0;
        const double ss = 1.0 / filterscale;
        int xmin = static_cast<int>(center - support + 0.5);
        if (xmin < 0) xmin = 0;
        int xmax = static_cast<int>(center + support + 0.5);
        if (xmax > in_size) xmax = in_size;
        xmax -= xmin;
        int x = 0;
        for (; x < xmax; ++x) {
            const double w = pil_bicubic((x + xmin - center + 0.5) * ss);
            k[x] = w;
            ww += w;
        }
        for (x = 0; x < xmax; ++x)
            if (ww != 0.0) k[x] /= ww;
        for (; x < ksize; ++x) k[x] = 0;
        for (x = 0; x < ksize; ++x) {
            const double v = k[x] * (1 << ub::kResizePrecisionBits);
            kk[static_cast<size_t>(xx) * ksize + x] = k[x] < 0 ? static_cast<int>(-0.5 + v) : static_cast<int>(0.5 + v);
        }
        bounds[2 * xx] = xmin;
        bounds[2 * xx + 1] = xmax;
    }
    return 0;
}

int unetb200_resize_bicubic_u8(const uint8_t* src, int n, int h, int w, int c, const int32_t* kx_dev,
                               const int32_t* bx_dev, int ksx, const int32_t* ky_dev, const int32_t* by_dev,
                               int ksy, uint8_t* tmp_dev, uint8_t* dst_dev, int oh, int ow, void* stream) {
    return unetb200_resize_bicubic_u8_ps(src, n, h, w, c, c, kx_dev, bx_dev, ksx, ky_dev, by_dev, ksy, tmp_dev,
                                         dst_dev, oh, ow, stream);
}

int unetb200_resize_bicubic_u8_ps(const uint8_t* src, int n, int h, int w, int c, int ps, const int32_t* kx_dev,
                                  const int32_t* bx_dev, int ksx, const int32_t* ky_dev, const int32_t* by_dev,
                                  int ksy, uint8_t* tmp_dev, uint8_t* dst_dev, int oh, int ow, void* stream) {
    if (!src || !dst_dev || n <= 0 || h <= 0 || w <= 0 || oh <= 0 || ow <= 0)
        return fail(UNETB200_EINVAL, "resize: bad argument");
    if (!(c == 1 || c == 3 || c == 4)) return fail(UNETB200_EINVAL, "resize: channels must be 1, 3 or 4");
    if (ps < c || ps > 16) return fail(UNETB200_EINVAL, "resize: pixel stride must be in [channels, 16]");
    const bool need_h = ow != w, need_v = oh != h;
    if (ps != c && !need_h)
        return fail(UNETB200_EINVAL, "resize: a padded source (pixel stride != channels) needs a horizontal pass");
    if (need_h && (!kx_dev || !bx_dev)) return fail(UNETB200_EINVAL, "resize: horizontal tables missing");
    if (need_v && (!ky_dev || !by_dev)) return fail(UNETB200_EINVAL, "resize: vertical tables missing");
    if (need_h && need_v && !tmp_dev) return fail(UNETB200_EINVAL, "resize: intermediate buffer missing");
    if (static_cast<long long>(n) * h > 2147483647LL || oh > 65535 || n > 65535)
        return fail(UNETB200_EINVAL, "resize: image too large");
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const uint8_t* cur = src;
    if (need_h) {
        uint8_t* out = need_v ? tmp_dev : dst_dev;
        dim3 grid((ow + 127) / 128, n * h);
        if (n * h > 65535) {
            // rows beyond the grid.y limit: one launch per image
            for (int i = 0; i < n; ++i) {
                dim3 g((ow + 127) / 128, h);
                const uint8_t* si = src + static_cast<size_t>(i) * h * w * ps;
                uint8_t* oi = out + static_cast<size_t>(i) * h * ow * c;
                if (c == 1) ub::resize_horizontal_kernel<1><<<g, 128, 0, s>>>(si, oi, kx_dev, bx_dev, ksx, h, w, ow, ps);
                else if (c == 3) ub::resize_horizontal_kernel<3><<<g, 128, 0, s>>>(si, oi, kx_dev, bx_dev, ksx, h, w, ow, ps);
                else ub::resize_horizontal_kernel<4><<<g, 128, 0, s>>>(si, oi, kx_dev, bx_dev, ksx, h, w, ow, ps);
            }
        } else if (c == 1) {
            ub::resize_horizontal_kernel<1><<<grid, 128, 0, s>>>(src, out, kx_dev, bx_dev, ksx, n * h, w, ow, ps);
        } else if (c == 3) {
            ub::resize_horizontal_kernel<3><<<grid, 128, 0, s>>>(src, out, kx_dev, bx_dev, ksx, n * h, w, ow, ps);
        } else {
            ub::resize_horizontal_kernel<4><<<grid, 128, 0, s>>>(src, out, kx_dev, bx_dev, ksx, n * h, w, ow, ps);
        }
        cur = out;
    }
    if (need_v) {
        const int wc = ow * c;
        dim3 grid((wc + 255) / 256, oh, n);
        ub::resize_vertical_kernel<<<grid, 256, 0, s>>>(cur, dst_dev, ky_dev, by_dev, ksy, h, oh, wc);
    } else if (!need_h) {
        UB_CUDA(cudaMemcpyAsync(dst_dev, src, static_cast<size_t>(n) * h * w * c, cudaMemcpyDeviceToDevice, s));
    }
    UB_CUDA(cudaGetLastError());
    return 0;
}

int unetb200_mask_bbox(const uint8_t* mask, int n_planes, int h, int w, int32_t* out, void* stream) {
    if (!mask || !out || n_planes <= 0 || h <= 0 || w <= 0) return fail(UNETB200_EINVAL, "mask_bbox: bad argument");
    ub::mask_bbox_kernel<<<n_planes, 256, 0, static_cast<cudaStream_t>(stream)>>>(mask, h, w, out);
    UB_CUDA(cudaGetLastError());
    return 0;
}

int unetb200_mask_bbox_bits(const uint8_t* bits, int n_planes, int h, int w, int32_t* out, void* stream) {
    if (!bits || !out || n_planes <= 0 || h <= 0 || w <= 0 || (w & 31) || (reinterpret_cast<uintptr_t>(bits) & 3))
        return fail(UNETB200_EINVAL, "mask_bbox_bits: bad argument (w must be a multiple of 32, bits 4-byte aligned)");
    ub::mask_bbox_bits_kernel<<<n_planes, 256, 0, static_cast<cudaStream_t>(stream)>>>(bits, h, w, out);
    UB_CUDA(cudaGetLastError());
    return 0;
}

// Host-side check of the kernels' division-by-launch-constant (conv_tc.cuh FastDiv): the quotient the
// device computes as __umulhi(x, mul) >> shr, evaluated here with the same magic numbers.
uint32_t unetb200_test_fastdiv(uint32_t d, uint32_t x) {
    if (d == 0) return 0xffffffffu;
    const ub::FastDiv f = ub::make_fastdiv(d);
    if (f.d == 1) return x;
    return static_cast<uint32_t>((static_cast<uint64_t>(x) * f.mul) >> 32) >> f.shr;
}

int unetb200_box_sums(const uint8_t* img, int h, int w, int c, const int32_t* boxes_host, int n_boxes,
                      uint64_t* sums_dev, void* stream) {
    return unetb200_box_sums_ps(img, h, w, c, c, boxes_host, n_boxes, sums_dev, stream);
}

int unetb200_box_sums_ps(const uint8_t* img, int h, int w, int c, int used, const int32_t* boxes_host, int n_boxes,
                         uint64_t* sums_dev, void* stream) {
    if (!img || !boxes_host || !sums_dev || h <= 0 || w <= 0 || c <= 0 || n_boxes <= 0 || n_boxes > ub::kMaxBoxes)
        return fail(UNETB200_EINVAL, "box_sums: bad argument");
    if (!(used == c || (c == 4 && used == 3 && (reinterpret_cast<uintptr_t>(img) & 3) == 0)))
        return fail(UNETB200_EINVAL, "box_sums: used bytes per pixel must equal the pixel size, or 3 of 4 (aligned RGBX)");
    ub::BoxList bl;
    bl.n = n_boxes;
    int rows = 1;
    for (int i = 0; i < n_boxes; ++i) {
        const int32_t* b = boxes_host + 4 * i;
        if (b[0] < 0 || b[1] < 0 || b[2] > w || b[3] > h || b[2] < b[0] || b[3] < b[1])
            return fail(UNETB200_EINVAL, "box_sums: rectangle outside the frame");
        bl.x1[i] = b[0]; bl.y1[i] = b[1]; bl.x2[i] = b[2]; bl.y2[i] = b[3];
        rows = std::max(rows, b[3] - b[1]);
    }
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    UB_CUDA(cudaMemsetAsync(sums_dev, 0, sizeof(uint64_t) * n_boxes, s));
    dim3 grid(static_cast<unsigned>(std::min(rows, 296)), static_cast<unsigned>(n_boxes));
    ub::box_sum_kernel<<<grid, 256, 0, s>>>(img, w, c, used, bl, reinterpret_cast<unsigned long long*>(sums_dev));
    UB_CUDA(cudaGetLastError());
    return UNETB200_OK;
}

}  // extern "C"
