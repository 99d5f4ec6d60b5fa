// Host launcher for the tcgen05 shift-GEMM convolution (kernel in conv_umma.cuh).
#include "sidekit_b200.h"
#include "conv_umma.cuh"
#include "conv3_umma.cuh"

#include <cstdlib>
#include "layers.cuh"

namespace skb {

int conv_pick_ncta(int cout) { return cout <= 32 ? 32 : (cout <= 64 ? 64 : 128); }
int conv_tile_m(int n_cta) { return n_cta == 32 ? 512 : 256; }
// N tiles whose plain epilogue can accumulate ConvParams::sums: one N split below 128 channels, at most two (ConvTotals) at 128
bool conv_sums_supported(int n_cta, int cout) { return n_cta == 128 ? (cout == 128 || cout == 256) : cout == n_cta; }

template <int N_CTA, int MT, bool BF16, bool FUSED, bool SC = false, bool TOT = false>
static int launch_one(const ConvParams& p_in, cudaStream_t st) {
    using Cfg = ConvCfg<N_CTA, MT, SC>;
    static PerDeviceOnce configured;
    ConvParams p = p_in;
    const size_t a_stage = (size_t)p.rows_pad * (kConvKC / 8) * 16;
    // Weights: resident for the life of the CTA when one N split's images fit in <= 96 KB (no per-item weight
    // traffic, no barrier round trips on the MMA issue path); otherwise streamed through a ring deep enough to
    // cover the L2 latency at the rate the MMAs consume them (the ring gets what the 3-slab A ring leaves).
    p.bias_mma = p.cout <= 256 ? 1 : 0;     // wide layers (TDNN) keep the epilogue bias add: their bias images would not fit
    // narrow layers keep the SE scale table (n_utt x cout floats) in shared memory: the epilogue's scale rows become
    // shared-memory reads instead of dependent L2 loads
    p.scale_smem_bytes = 0;
    if (FUSED && N_CTA <= 64 && (size_t)p.n_utt * p.cout * 4 <= 32 * 1024) p.scale_smem_bytes = p.n_utt * p.cout * 4;
    const int scb = p.scale_smem_bytes;
    if (!SC) p.sc_cin = 0;
    const int n_it = p.n_pairs;
    const int n_split = p.cout / N_CTA;
    int tps = 1, bst = 1;
    p.b_resident = (n_split == 1 && (size_t)n_it * Cfg::kBStageBytes <= 96 * 1024) ? 1 : 0;
    size_t b_stage = Cfg::kBStageBytes;
    if (p.b_resident) {
        bst = n_it;
    } else {
        if (p.kc_per_grp == p.cin / kConvKC) {      // single tap group: several taps per weight stage
            for (int cand : {3, 5}) {
                if (p.taps % cand == 0 && (size_t)cand * Cfg::kBStageBytes <= 24 * 1024) { tps = cand; break; }
            }
        }
        b_stage = (size_t)tps * Cfg::kBStageBytes;
        const size_t left = kConvSmemBudget - Cfg::fixed_bytes(p.cout, p.bias_mma, 0, 0, scb, p.sc_cin, TOT) - 3 * a_stage;
        bst = (int)(left / b_stage);
        if (bst > kConvBStages) bst = kConvBStages;
        if (bst < 2) bst = 2;
    }
    p.tps = tps;
    p.b_stages = bst;
    const size_t fixed = Cfg::fixed_bytes(p.cout, p.bias_mma, bst, tps, scb, p.sc_cin, TOT);
    int stages = (int)((kConvSmemBudget - fixed) / a_stage);
    if (stages > kConvMaxAStages) stages = kConvMaxAStages;
    if (stages < 2) {
        set_last_error(__FILE__, __LINE__, "conv slab does not fit in shared memory");
        return SKB_ERR_ARG;
    }
    p.a_stages = stages;
    const size_t smem = fixed + (size_t)stages * a_stage;
    if (configured.first()) {
        SKB_CUDA_CHECK(cudaFuncSetAttribute(conv_umma_kernel<N_CTA, MT, BF16, FUSED, SC, TOT>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                            227 * 1024));
    }
    const int n_pix = p.p_end - p.G;
    p.n_tiles = (n_pix + Cfg::kTileM - 1) / Cfg::kTileM;
    const int n_items = p.n_tiles * (p.cout / N_CTA);
    const int grid = n_items < kNumSMs ? n_items : kNumSMs;      // persistent: one CTA per SM
    SKB_CUDA_CHECK(launch_kernel(true, conv_umma_kernel<N_CTA, MT, BF16, FUSED, SC, TOT>, dim3(grid), dim3(kConvThreads), smem, st, p));
    return SKB_OK;
}

// Fused-tap kernel for the narrow 3x3 / stride-1 convolutions (conv3_umma.cuh).
template <int N_CTA, int MT, bool BF16>
static int launch_one3(const ConvParams& p_in, cudaStream_t st) {
    using Cfg = Conv3Cfg<N_CTA, MT>;
    static PerDeviceOnce configured;
    ConvParams p = p_in;
    p.halo = p.Wp;                                          // one line above / below; the +-1 pixel shifts happen in the epilogue
    p.rows_pad = (Cfg::kTileM + 2 * p.Wp + 7) / 8 * 8;
    const int n_kc = p.cin / kConvKC;
    const size_t a_stage = (size_t)p.rows_pad * (kConvKC / 8) * 16;
    p.scale_smem_bytes = 0;
    if (p.se_scale != nullptr && (size_t)p.n_utt * N_CTA * 4 <= 32 * 1024) p.scale_smem_bytes = p.n_utt * N_CTA * 4;
    const size_t fixed = Cfg::fixed_bytes(n_kc, p.scale_smem_bytes);
    if (fixed + 2 * a_stage > (size_t)kConvSmemBudget || p.G < p.Wp + 1) {
        set_last_error(__FILE__, __LINE__, "fused-tap conv does not fit (shared memory or guard)");
        return SKB_ERR_ARG;
    }
    int stages = (int)((kConvSmemBudget - fixed) / a_stage);
    if (stages > kConvMaxAStages) stages = kConvMaxAStages;
    p.a_stages = stages;
    const size_t smem = fixed + (size_t)stages * a_stage;
    if (configured.first()) {
        SKB_CUDA_CHECK(cudaFuncSetAttribute(conv3_umma_kernel<N_CTA, MT, BF16>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    }
    const int n_pix = p.p_end - p.G;
    p.n_tiles = (n_pix + Cfg::kTileOut - 1) / Cfg::kTileOut;
    const int grid = p.n_tiles < kNumSMs ? p.n_tiles : kNumSMs;
    SKB_CUDA_CHECK(launch_kernel(false, conv3_umma_kernel<N_CTA, MT, BF16>, grid, kConvThreads, smem, st, p));
    return SKB_OK;
}

int launch_conv_umma(const ConvParams& p, int n_cta, bool bf16, cudaStream_t st) {
    // EXPERIMENTAL, off by default (SKB_FUSED_TAPS=1 enables it): parity-green, and its MMA loop is 2.4x / 1.5x shorter on
    // layers 1 / 2, but the lane-shifted epilogue (64 shuffles + 6 TMEM loads per 32 x 32 block) costs more than the MMAs
    // it saves: 417 / 230 us per launch against 295 / 178 us for conv_umma_kernel (profiles/r01c_fused_taps.txt).
    static const bool fused_taps = [] { const char* e = getenv("SKB_FUSED_TAPS"); return e && e[0] == '1'; }();
    // (the fused-tap kernel has no channel totals in its epilogue)
    if (p.w3 != nullptr && fused_taps && p.sc_in == nullptr && p.sums == nullptr && p.cout == n_cta && p.taps == 9 && p.cin % kConvKC == 0) {
        if (n_cta == 32) return bf16 ? launch_one3<32, 2, true>(p, st) : launch_one3<32, 2, false>(p, st);
        if (n_cta == 64) return bf16 ? launch_one3<64, 1, true>(p, st) : launch_one3<64, 1, false>(p, st);
    }
    if (p.cin % kConvKC != 0 || p.cout % n_cta != 0 || p.taps < 1 || p.taps > 10 || p.rows_pad % 8 != 0 || p.kc_per_grp < 1 || p.n_pairs < 1) {
        set_last_error(__FILE__, __LINE__, "conv_umma: unsupported shape");
        return SKB_ERR_ARG;
    }
    const bool fused = p.se_scale != nullptr;
    if (p.sums != nullptr && (fused || p.sc_in != nullptr || p.pix_sub != nullptr || !conv_sums_supported(n_cta, p.cout))) {
        set_last_error(__FILE__, __LINE__, "conv_umma: channel totals unsupported for this shape");
        return SKB_ERR_ARG;
    }
    if (p.sc_in != nullptr) {
        // folded shortcut: the narrow layers only (the <128, 2> tiles already use all 512 TMEM columns)
        if (!fused || p.sc_w == nullptr || p.sc_bias == nullptr || p.sc_cin < kConvKC || p.sc_cin % kConvKC != 0 || p.cout > 256) {
            set_last_error(__FILE__, __LINE__, "conv_umma: unsupported folded shortcut");
            return SKB_ERR_ARG;
        }
        if (n_cta == 32) return bf16 ? launch_one<32, 4, true, true, true>(p, st) : launch_one<32, 4, false, true, true>(p, st);
        if (n_cta == 64) return bf16 ? launch_one<64, 2, true, true, true>(p, st) : launch_one<64, 2, false, true, true>(p, st);
        set_last_error(__FILE__, __LINE__, "conv_umma: folded shortcut needs an N tile of 32 or 64");
        return SKB_ERR_ARG;
    }
#define SKB_CONV_CASE(N, M)                                                                                   \
    case N:                                                                                                   \
        if (fused) return bf16 ? launch_one<N, M, true, true>(p, st) : launch_one<N, M, false, true>(p, st);  \
        return bf16 ? launch_one<N, M, true, false>(p, st) : launch_one<N, M, false, false>(p, st);
    if (p.sums != nullptr && n_cta == 64)
        return bf16 ? launch_one<64, 2, true, false, false, true>(p, st) : launch_one<64, 2, false, false, false, true>(p, st);
    if (p.sums != nullptr && n_cta == 128)
        return bf16 ? launch_one<128, 2, true, false, false, true>(p, st) : launch_one<128, 2, false, false, false, true>(p, st);
    switch (n_cta) {
        SKB_CONV_CASE(32, 4)
        SKB_CONV_CASE(64, 2)
        SKB_CONV_CASE(128, 2)
    }
#undef SKB_CONV_CASE
    set_last_error(__FILE__, __LINE__, "conv_umma: unsupported N tile");
    return SKB_ERR_ARG;
}

}  // namespace skb
