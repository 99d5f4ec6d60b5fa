// Memory-bound and small kernels around the tcgen05 convolutions: stem conv, squeeze-excitation,
// residual merge, statistics / attentive pooling, the embedding head, and an fp32 SIMT GEMM for the
// small dense layers.  All operate on the chunk-plane activation layout described in conv_umma.cuh.
#include "sidekit_b200.h"
#include "common.cuh"
#include "layers.cuh"

namespace skb {

// ----------------------------------------------------------------------------- stem: 3x3 conv 1->32 + BN + ReLU
// sidekit/nnet/res_net.py:549 (relu(bn1(conv1(x)))) on the (B,1,T,F) view of the features.
// One thread per kStemPix level-1 pixels; the normalised features are frame-major so a warp reads contiguous
// mel bins.  fp32 math on CUDA cores (0.1 % of the trunk's FLOPs), 16-bit chunk-plane output.
constexpr int kStemPix = 2;            // pixels per thread
template <bool BF16, int COUT>
__global__ void __launch_bounds__(128) stem_kernel(const __grid_constant__ StemConsts sc, const float* __restrict__ feats,
                                                   const long long* __restrict__ feat_off, const int* __restrict__ n_frames,
                                                   const float2* __restrict__ cmvn /*[B][W] (mean, rstd)*/,
                                                   uint16_t* __restrict__ out, long long out_plane, int G, int p_end, int Wp,
                                                   int W, const int* __restrict__ row_b, const int* __restrict__ row_h,
                                                   unsigned* __restrict__ overflow) {
    uint32_t omax = 0u;                    // fp16 range guard (common.cuh)
    // The folded weights arrive as a kernel parameter: every FFMA takes its weight straight from the constant bank
    // (a shared-memory copy costs one LDS per FMA and made the kernel LSU-bound at 3x its HBM time).  Each thread computes
    // kStemPix pixels (blockDim apart, so loads and stores stay coalesced): a weight fetched into a uniform register feeds
    // kStemPix FMAs (one pixel per thread spent a quarter of its 840 instructions per pixel on those fetches).
    const int pix0 = G + blockIdx.x * (blockDim.x * kStemPix) + threadIdx.x;
    float x[kStemPix][9];
    bool valid[kStemPix];
#pragma unroll
    for (int q = 0; q < kStemPix; ++q) {
        const int pix = pix0 + q * blockDim.x;
#pragma unroll
        for (int k = 0; k < 9; ++k) x[q][k] = 0.f;
        valid[q] = false;
        if (pix >= p_end) continue;
        const int rel = pix - G;
        const int row = rel / Wp, f = rel - row * Wp;
        const int b = row_b[row], t = row_h[row];
        valid[q] = (b >= 0) && (f < W);
        if (valid[q]) {
            const int T = n_frames[b];
            const float* fb = feats + (size_t)feat_off[b] * W;
#pragma unroll
            for (int df = 0; df < 3; ++df) {
                const int ff = f + df - 1;
                const bool f_ok = ff >= 0 && ff < W;
                // CMVN (InstanceNorm1d) applied on the fly to the raw log-Mel features: (x - mean) * rstd per (utterance, bin)
                const float2 ms = f_ok ? __ldg(cmvn + (size_t)b * W + ff) : make_float2(0.f, 0.f);
#pragma unroll
                for (int dt = 0; dt < 3; ++dt) {
                    const int tt = t + dt - 1;
                    x[q][dt * 3 + df] = (f_ok && tt >= 0 && tt < T) ? (__ldg(fb + (size_t)tt * W + ff) - ms.x) * ms.y : 0.f;
                }
            }
        }
    }
#pragma unroll
    for (int g = 0; g < COUT / 8; ++g) {           // 8 output channels (one 16-byte chunk) at a time, for every pixel of the thread
        float acc[kStemPix][8];
#pragma unroll
        for (int c = 0; c < 8; ++c) {
            float a[kStemPix];
#pragma unroll
            for (int q = 0; q < kStemPix; ++q) a[q] = sc.b[g * 8 + c];
#pragma unroll
            for (int k = 0; k < 9; ++k) {
                const float w = sc.w[(g * 8 + c) * 9 + k];
#pragma unroll
                for (int q = 0; q < kStemPix; ++q) a[q] = fmaf(w, x[q][k], a[q]);
            }
#pragma unroll
            for (int q = 0; q < kStemPix; ++q) acc[q][c] = valid[q] ? fmaxf(a[q], 0.f) : 0.f;
        }
#pragma unroll
        for (int q = 0; q < kStemPix; ++q) {
            const int pix = pix0 + q * blockDim.x;
            if (pix >= p_end) continue;
            uint4 o;
            o.x = pack2<BF16>(acc[q][0], acc[q][1]);
            o.y = pack2<BF16>(acc[q][2], acc[q][3]);
            o.z = pack2<BF16>(acc[q][4], acc[q][5]);
            o.w = pack2<BF16>(acc[q][6], acc[q][7]);
            *reinterpret_cast<uint4*>(out + ((size_t)g * out_plane + pix) * 8) = o;
            if (!BF16) track16(o, omax);
        }
    }
    if (!BF16 && overflow != nullptr && saturated16(omax)) atomicAdd(overflow, 1u);
}

int launch_stem(bool bf16, int cout, const float* feats, const long long* feat_off, const int* n_frames, const float2* cmvn,
                const StemConsts& sc, uint16_t* out, long long out_plane, int G, int p_end, int Wp, int W,
                const int* row_b, const int* row_h, unsigned* overflow, cudaStream_t st) {
    const int n = p_end - G;
    const int threads = 128;
    const int blocks = (n + threads * kStemPix - 1) / (threads * kStemPix);
    if (cout != 32 && cout != 128) {
        set_last_error(__FILE__, __LINE__, "stem: 32 or 128 output channels");
        return SKB_ERR_ARG;
    }
    const auto kernel = cout == 32 ? (bf16 ? stem_kernel<true, 32> : stem_kernel<false, 32>)
                                   : (bf16 ? stem_kernel<true, 128> : stem_kernel<false, 128>);
    SKB_CUDA_CHECK(launch_kernel(false, kernel, blocks, threads, 0, st, sc, feats, feat_off, n_frames, cmvn, out, out_plane, G, p_end, Wp, W, row_b,
                                 row_h, overflow));
    return SKB_OK;
}

// ----------------------------------------------------------------------------- fastresnet34 stem: 7x7 conv 1->16, stride (1, 2)
// sidekit/nnet/res_net.py:566-572, :605: relu(bn1(conv1(x))) on the (B,1,T,F=80) view, padding 3, stride 1 along time and 2
// along frequency -> (B,16,T,40).  One thread per output pixel; the 16 real channels are written as chunks 0-1 and the
// level is carried with 32 channels (chunks 2-3 = 0) so that the K = 32 tensor-core convolutions need no special case.
template <bool BF16>
__global__ void __launch_bounds__(128) stem7_kernel(const __grid_constant__ StemConsts sc, const float* __restrict__ feats,
                                                    const long long* __restrict__ feat_off, const int* __restrict__ n_frames,
                                                    const float2* __restrict__ cmvn /*[B][F] (mean, rstd)*/,
                                                    uint16_t* __restrict__ out, long long out_plane, int G, int p_end, int Wp,
                                                    int W, int F, const int* __restrict__ row_b, const int* __restrict__ row_h,
                                                    unsigned* __restrict__ overflow) {
    const int pix = G + blockIdx.x * blockDim.x + threadIdx.x;
    if (pix >= p_end) return;
    const int rel = pix - G;
    const int row = rel / Wp, wo = rel - row * Wp;
    const int b = row_b[row], t = row_h[row];
    const bool valid = (b >= 0) && (wo < W);
    float acc[16];
#pragma unroll
    for (int c = 0; c < 16; ++c) acc[c] = sc.b[c];
    if (valid) {
        const int T = n_frames[b];
        const float* fb = feats + (size_t)feat_off[b] * F;
#pragma unroll
        for (int s = 0; s < 7; ++s) {
            const int ff = 2 * wo + s - 3;
            if (ff < 0 || ff >= F) continue;
            const float2 ms = __ldg(cmvn + (size_t)b * F + ff);
#pragma unroll
            for (int r = 0; r < 7; ++r) {
                const int tt = t + r - 3;
                if (tt < 0 || tt >= T) continue;
                const float x = (__ldg(fb + (size_t)tt * F + ff) - ms.x) * ms.y;
#pragma unroll
                for (int c = 0; c < 16; ++c) acc[c] = fmaf(sc.w[c * 49 + r * 7 + s], x, acc[c]);
            }
        }
    }
#pragma unroll
    for (int c = 0; c < 16; ++c) acc[c] = valid ? fmaxf(acc[c], 0.f) : 0.f;
    uint32_t omax = 0u;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        uint4 o = make_uint4(0u, 0u, 0u, 0u);
        if (j < 2) {
            o.x = pack2<BF16>(acc[j * 8 + 0], acc[j * 8 + 1]);
            o.y = pack2<BF16>(acc[j * 8 + 2], acc[j * 8 + 3]);
            o.z = pack2<BF16>(acc[j * 8 + 4], acc[j * 8 + 5]);
            o.w = pack2<BF16>(acc[j * 8 + 6], acc[j * 8 + 7]);
            if (!BF16) track16(o, omax);
        }
        *reinterpret_cast<uint4*>(out + ((size_t)j * out_plane + pix) * 8) = o;
    }
    if (!BF16 && overflow != nullptr && saturated16(omax)) atomicAdd(overflow, 1u);
}

int launch_stem7(bool bf16, const float* feats, const long long* feat_off, const int* n_frames, const float2* cmvn,
                 const StemConsts& sc, uint16_t* out, long long out_plane, int G, int p_end, int Wp, int W, int F,
                 const int* row_b, const int* row_h, unsigned* overflow, cudaStream_t st) {
    const int n = p_end - G;
    const int threads = 128;
    const int blocks = (n + threads - 1) / threads;
    SKB_CUDA_CHECK(launch_kernel(false, bf16 ? stem7_kernel<true> : stem7_kernel<false>, blocks, threads, 0, st, sc, feats, feat_off, n_frames, cmvn,
                                 out, out_plane, G, p_end, Wp, W, F, row_b, row_h, overflow));
    return SKB_OK;
}

// out[b][a] = bias[a]: the per-utterance attention bias when the pooling has no global context
__global__ void broadcast_rows_kernel(const float* __restrict__ bias, int B, int A, float* __restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < B * A) out[i] = bias[i % A];
}

int launch_broadcast_rows(const float* bias, int B, int A, float* out, cudaStream_t st) {
    SKB_CUDA_CHECK(launch_kernel(false, broadcast_rows_kernel, (B * A + 255) / 256, 256, 0, st, bias, B, A, out));
    return SKB_OK;
}

// ----------------------------------------------------------------------------- SE squeeze, computed BEFORE conv2 runs
// The SE layer needs mean_{h,w}(bn2(conv2(y1))) per (utterance, channel) (sidekit/nnet/res_net.py:272-281, :316-317).
// conv2 is linear, so that mean follows from sums of its INPUT y1:
//     sum_{h,w} y2[c] = N*b2[c] + sum_{tap,ci} W2[c][ci][tap] * S_tap[ci],
//     S_(dr,ds)[ci] = Total[ci] - (excluded border row) - (excluded border column) + (their corner)
// (a tap shifted by (dr, ds) sees every pixel except one border row / column; the zero padding contributes nothing).
// Knowing the scales up front lets conv2's epilogue apply scale + residual + ReLU directly: y2 is never stored and
// the separate "scale, add, ReLU" pass disappears.
//
// plane_sum_kernel: Total[b][ci] over the valid pixels, in 2^-15 FIXED POINT (each 16-bit activation is rounded to a
// multiple of 2^-15 -- a pure function of the pixel -- and integer addition is associative), so the sums, and through
// them every embedding, are bit-identical whatever the packing, grid shape or atomic order.
// One warp per 256-pixel span and chunk plane.  A per-span table (span_b: the utterance when every valid pixel of the
// span belongs to one, -1 when the span holds only pad pixels, -2 when it straddles utterances) replaces the per-pixel
// utterance lookups, so the common path is eight independent 16-byte loads per lane followed by the arithmetic (the
// first version looked up pix_b before every load: one load in flight per thread, 50 % of the HBM roofline).  Pad
// pixels hold zeros and are simply added.
constexpr float kSeFixScale = 32768.f;          // 2^15: |x| <= 65504 still fits a signed 32-bit integer
constexpr double kSeFixInv = 1.0 / 32768.0;
constexpr int kSpanPix = 256;

template <bool BF16>
__device__ __forceinline__ void fix_add8(const uint4& a, long long (&t)[8]) {
    const uint32_t u[4] = {a.x, a.y, a.z, a.w};
#pragma unroll
    for (int e = 0; e < 4; ++e) {
        float2 v = unpack2<BF16>(u[e]);
        if (BF16) { v.x = fminf(fmaxf(v.x, -65504.f), 65504.f); v.y = fminf(fmaxf(v.y, -65504.f), 65504.f); }
        t[2 * e] += (long long)__float2int_rn(v.x * kSeFixScale);
        t[2 * e + 1] += (long long)__float2int_rn(v.y * kSeFixScale);
    }
}

// Exact warp sums of eight 64-bit values: a shuffle transpose-reduce (each step halves the values a lane carries), 18
// 64-bit shuffles in all.  Lane l ends up with the total of value e = 4*b4 + 2*b3 + b2 (bits of l); the result is
// returned by the lanes with b1 = b0 = 0, i.e. lane 4*e' ... see `sum8_slot`.  __reduce_add_sync (REDUX) measured
// ~20 cycles per instruction per SM here and made this kernel REDUX-bound on the small levels.
__device__ __forceinline__ int sum8_slot(int lane) { return ((lane >> 4) & 1) * 4 + ((lane >> 3) & 1) * 2 + ((lane >> 2) & 1); }
__device__ __forceinline__ long long warp_sum8_i64(const long long (&t)[8], int lane) {
    long long v[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) v[e] = t[e];
#pragma unroll
    for (int step = 0; step < 3; ++step) {               // offsets 16, 8, 4: keep 4, 2, 1 values
        const int off = 16 >> step, keep = 4 >> step;
        const bool upper = (lane & off) != 0;
#pragma unroll
        for (int i = 0; i < keep; ++i) {
            const long long send = upper ? v[i] : v[i + keep];
            const long long mine = upper ? v[i + keep] : v[i];
            v[i] = mine + shfl_xor_ll(send, off);
        }
    }
    v[0] += shfl_xor_ll(v[0], 2);
    v[0] += shfl_xor_ll(v[0], 1);
    return v[0];                                          // total of value sum8_slot(lane), replicated over 4 lanes
}

template <bool BF16>
__device__ __forceinline__ void plane_sum_body(const uint16_t* __restrict__ act, long long plane, int G, int p_end,
                                               const int* __restrict__ pix_b, const int* __restrict__ span_b, int C,
                                               int planes_per_block, unsigned long long* __restrict__ sums) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int span = blockIdx.x * 8 + warp;
    const int base = G + span * kSpanPix;
    if (base >= p_end) return;
    const int sb = __ldg(span_b + span);
    if (sb == -1) return;                                  // pad pixels only: all zeros
    const int j0 = blockIdx.y * planes_per_block;
    int pb[8];                                             // per-pixel utterances, only needed when the span is mixed
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        pb[k] = -1;
        if (sb == -2 && base + k * 32 + lane < p_end) pb[k] = __ldg(pix_b + (base + k * 32 + lane - G));
    }
    for (int j = j0; j < j0 + planes_per_block; ++j) {
        const uint16_t* src = act + ((size_t)j * plane + base + lane) * 8;
        uint4 a[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            a[k] = make_uint4(0u, 0u, 0u, 0u);
            if (base + k * 32 + lane < p_end) a[k] = *reinterpret_cast<const uint4*>(src + (size_t)k * 32 * 8);
        }
        if (sb >= 0) {
            long long t[8];
#pragma unroll
            for (int e = 0; e < 8; ++e) t[e] = 0ll;
#pragma unroll
            for (int k = 0; k < 8; ++k) fix_add8<BF16>(a[k], t);
            const long long mine = warp_sum8_i64(t, lane);
            if ((lane & 3) == 0) atomicAdd(sums + (size_t)sb * C + j * 8 + sum8_slot(lane), (unsigned long long)mine);
        } else {
            // the span straddles utterance boundaries (the rule on the deepest level, where an utterance is a few hundred
            // pixels): one warp-uniform pass per distinct utterance, in increasing order
            int cur = -1;
            while (true) {
                int mine_b = 0x7fffffff;
#pragma unroll
                for (int k = 0; k < 8; ++k)
                    if (pb[k] > cur) mine_b = min(mine_b, pb[k]);
                const int nb = __reduce_min_sync(0xffffffffu, mine_b);
                if (nb == 0x7fffffff) break;
                long long t[8];
#pragma unroll
                for (int e = 0; e < 8; ++e) t[e] = 0ll;
#pragma unroll
                for (int k = 0; k < 8; ++k)
                    if (pb[k] == nb) fix_add8<BF16>(a[k], t);
                const long long mine = warp_sum8_i64(t, lane);
                if ((lane & 3) == 0) atomicAdd(sums + (size_t)nb * C + j * 8 + sum8_slot(lane), (unsigned long long)mine);
                cur = nb;
            }
        }
    }
}

// The previous kernel of the stream is se_border_kernel, which waited for conv1 BEFORE it let this grid start and whose
// results this kernel does not use -- so the sums start at once, beside the border CTAs, and the wait is at the end (this
// grid must not complete before the border grid: the kernel after it waits for this one only).
template <bool BF16>
__global__ void __launch_bounds__(256, 4) plane_sum_kernel(const uint16_t* __restrict__ act, long long plane, int G, int p_end,
                                                        const int* __restrict__ pix_b, const int* __restrict__ span_b, int C,
                                                        int planes_per_block, unsigned long long* __restrict__ sums) {
    plane_sum_body<BF16>(act, plane, G, p_end, pix_b, span_b, C, planes_per_block, sums);
    pdl_wait();
}

// span_b table for plane_sum_kernel (built once per batch composition)
__global__ void span_table_kernel(const int* __restrict__ pix_b, int n, int n_spans, int* __restrict__ span_b) {
    const int span = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (span >= n_spans) return;
    int mn = 0x7fffffff, mx = -1;
    for (int k = 0; k < kSpanPix / 32; ++k) {
        const int rel = span * kSpanPix + k * 32 + lane;
        const int b = rel < n ? pix_b[rel] : -1;
        if (b >= 0) { mn = min(mn, b); mx = max(mx, b); }
    }
    mn = __reduce_min_sync(0xffffffffu, mn);
    mx = __reduce_max_sync(0xffffffffu, mx);
    if (lane == 0) span_b[span] = mx < 0 ? -1 : (mn == mx ? mn : -2);
}

int span_table_size(int n_pix) { return (n_pix + kSpanPix - 1) / kSpanPix; }

int launch_span_table(const int* pix_b, int n_pix, int* span_b, cudaStream_t st) {
    const int n_spans = span_table_size(n_pix);
    SKB_CUDA_CHECK(launch_kernel(false, span_table_kernel, (n_spans + 7) / 8, 256, 0, st, pix_b, n_pix, n_spans, span_b));
    return SKB_OK;
}

static int launch_plane_sum(bool bf16, const uint16_t* act, long long plane, int G, int p_end, const int* pix_b, const int* span_b,
                            int C, unsigned long long* sums, cudaStream_t st) {
    const int n = p_end - G;
    const int n_spans = span_table_size(n);
    const int chunks = C / 8;
    const int ppb = chunks >= 16 ? 4 : (chunks >= 8 ? 2 : 1);      // keep >= ~4 waves of CTAs on the small levels
    dim3 grid((n_spans + 7) / 8, chunks / ppb);
    SKB_CUDA_CHECK(launch_kernel(true, bf16 ? plane_sum_kernel<true> : plane_sum_kernel<false>, grid, dim3(256), 0, st, act, plane, G, p_end, pix_b,
                                 span_b, C, ppb, sums));
    return SKB_OK;
}

// se_border_kernel: sums of the first / last row and column of y1 and its four corner pixels, per (utterance, channel).
// One CTA per (utterance, 8-channel chunk); threads stride over the border pixels with 16-byte loads; the block
// reduction runs in a fixed order, so the result is deterministic.  brd layout: [B][8 kinds][C].
template <bool BF16>
__global__ void __launch_bounds__(256) se_border_kernel(const uint16_t* __restrict__ y1, long long plane, int G, int Wp, int W,
                                                        const int* __restrict__ utt_row0, const int* __restrict__ utt_count, int C,
                                                        float* __restrict__ brd) {
    __shared__ float part[256][33];
    __shared__ float part2[8][32];
    pdl_wait();
    pdl_trigger_now();                              // conv1 is complete: the channel-total pass may start beside this grid
    const int b = blockIdx.x, j = blockIdx.y;
    const int H = utt_count[b] / W;
    const uint16_t* base = y1 + ((size_t)j * plane + G + (size_t)utt_row0[b] * Wp) * 8;     // pixel (0, 0) of chunk j
    float acc[32];                                  // [row0 | rowL | col0 | colL][8 channels]
#pragma unroll
    for (int i = 0; i < 32; ++i) acc[i] = 0.f;
    auto add8 = [&](const uint16_t* p, int o) {
        const uint4 a = *reinterpret_cast<const uint4*>(p);
        const uint32_t u[4] = {a.x, a.y, a.z, a.w};
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const float2 v = unpack2<BF16>(u[e]);
            acc[o + 2 * e] += v.x;
            acc[o + 2 * e + 1] += v.y;
        }
    };
    for (int w = threadIdx.x; w < W; w += blockDim.x) {
        add8(base + (size_t)w * 8, 0);
        add8(base + ((size_t)(H - 1) * Wp + w) * 8, 8);
    }
    // unrolled: the loads of four column pixels are in flight together (the rolled loop paid one L2 round trip each)
    for (int hh0 = threadIdx.x; hh0 < H; hh0 += 4 * blockDim.x) {
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int hh = hh0 + u * blockDim.x;
            if (hh < H) {
                add8(base + (size_t)hh * Wp * 8, 16);
                add8(base + ((size_t)hh * Wp + W - 1) * 8, 24);
            }
        }
    }
    // fixed-order two-level reduction through shared memory: thread (g, i) adds quantity i over partials 32g .. 32g+31,
    // then thread i adds the eight group totals
#pragma unroll
    for (int i = 0; i < 32; ++i) part[threadIdx.x][i] = acc[i];
    __syncthreads();
    {
        const int i = threadIdx.x & 31, g = threadIdx.x >> 5;
        float a = 0.f;
        for (int t = 0; t < 32; ++t) a += part[g * 32 + t][i];
        part2[g][i] = a;
    }
    __syncthreads();
    if (threadIdx.x < 32) {
        float a = 0.f;
        for (int t = 0; t < 8; ++t) a += part2[t][threadIdx.x];
        const int kind = threadIdx.x >> 3, e = threadIdx.x & 7;
        brd[((size_t)b * 8 + kind) * C + j * 8 + e] = a;
    }
    if (threadIdx.x >= 32 && threadIdx.x < 64) {    // corners: (0,0) (0,W-1) (H-1,0) (H-1,W-1)
        const int k = (threadIdx.x - 32) >> 3, e = threadIdx.x & 7;
        const int hh = (k >> 1) ? H - 1 : 0, ww = (k & 1) ? W - 1 : 0;
        const uint16_t u = base[((size_t)hh * Wp + ww) * 8 + e];
        brd[((size_t)b * 8 + 4 + k) * C + j * 8 + e] = unpack2<BF16>((uint32_t)u).x;
    }
}

// se_mean_partial_kernel: the mean of conv2's output through the (16-bit-rounded, BN-folded) conv2 weights, as a small
// GEMM  partial[ks][b][co] = sum_{i in K-slice ks} W2t[i][co] * S[b][i],  i = ci * 9 + tap,  S = the nine shifted sums.
// Grid = (Cin / 8 slices of 8 channels x 9 taps, utterance groups of 16); every weight row is read once per utterance
// group.  Fixed summation order everywhere -> deterministic.
constexpr int kSeCh = 8, kSeRows = 9 * kSeCh, kSeUtt = 16;
template <int Cout>
__global__ void __launch_bounds__(256) se_mean_partial_kernel(const unsigned long long* __restrict__ sums, const float* __restrict__ brd,
                                                              int B, int Cin, const float* __restrict__ w2t,
                                                              float* __restrict__ partial) {
    __shared__ float sS[kSeUtt][kSeRows];
    constexpr int n_rg = 256 / Cout;               // row groups: 8 / 4 / 2 / 1 for Cout = 32 / 64 / 128 / 256
    constexpr int RPT = kSeRows / n_rg;            // weight rows per thread: 9 / 18 / 36 / 72
    // this thread's weights first: RPT independent loads whose latency overlaps the shifted-sum phase below
    const int co = threadIdx.x % Cout, rg = threadIdx.x / Cout;
    float wreg[RPT];
    {
        const float* wp = w2t + ((size_t)blockIdx.x * kSeRows + rg) * Cout + co;
#pragma unroll
        for (int i = 0; i < RPT; ++i) wreg[i] = __ldg(wp + (size_t)i * n_rg * Cout);
    }
    pdl_wait();                                    // the weight loads above are constants: they overlap the previous kernel
    const int k0 = blockIdx.x * kSeRows, b0 = blockIdx.y * kSeUtt;
    const int nu = min(kSeUtt, B - b0);
    // the nine shifted sums of one (utterance, input channel): nine independent loads, then arithmetic only
    for (int idx = threadIdx.x; idx < kSeUtt * kSeCh; idx += blockDim.x) {
        const int u = idx / kSeCh, cl = idx - u * kSeCh;
        float v[9];
#pragma unroll
        for (int tap = 0; tap < 9; ++tap) v[tap] = 0.f;
        if (u < nu) {
            const int b = b0 + u, c = blockIdx.x * kSeCh + cl;
            const float* bb = brd + (size_t)b * 8 * Cin + c;
            const float tot = (float)((double)(long long)sums[(size_t)b * Cin + c] * kSeFixInv);
            const float row0 = bb[0], rowL = bb[Cin], col0 = bb[2 * Cin], colL = bb[3 * Cin];
            const float k00 = bb[4 * Cin], k0L = bb[5 * Cin], kL0 = bb[6 * Cin], kLL = bb[7 * Cin];
#pragma unroll
            for (int tap = 0; tap < 9; ++tap) {
                const int dr = tap / 3 - 1, ds = tap % 3 - 1;
                float x = tot;
                if (dr < 0) x -= rowL;                 // shifted up: the last row is never read
                if (dr > 0) x -= row0;
                if (ds < 0) x -= colL;
                if (ds > 0) x -= col0;
                if (dr < 0 && ds < 0) x += kLL;
                if (dr < 0 && ds > 0) x += kL0;
                if (dr > 0 && ds < 0) x += k0L;
                if (dr > 0 && ds > 0) x += k00;
                v[tap] = x;
            }
        }
#pragma unroll
        for (int tap = 0; tap < 9; ++tap) sS[u][cl * 9 + tap] = v[tap];
    }
    __syncthreads();
    // thread = (output channel co, row group rg): the 256 threads split the slice's rows so that even the 32-channel
    // layers keep 8 warps busy (one warp walking 64 dependent L2 loads was 45 us per launch); the row groups are then
    // added in a fixed order.
    __shared__ float sRed[256 * kSeUtt];
    float acc[kSeUtt];
#pragma unroll
    for (int u = 0; u < kSeUtt; ++u) acc[u] = 0.f;
#pragma unroll
    for (int i = 0; i < RPT; ++i) {
        const int r = rg + i * n_rg;
#pragma unroll
        for (int u = 0; u < kSeUtt; ++u) acc[u] = fmaf(wreg[i], sS[u][r], acc[u]);
    }
#pragma unroll
    for (int u = 0; u < kSeUtt; ++u) sRed[(rg * kSeUtt + u) * Cout + co] = acc[u];
    __syncthreads();
    for (int idx = threadIdx.x; idx < nu * Cout; idx += blockDim.x) {
        const int u = idx / Cout, c = idx - u * Cout;
        float a = 0.f;
        for (int g = 0; g < n_rg; ++g) a += sRed[(g * kSeUtt + u) * Cout + c];
        partial[((size_t)blockIdx.x * B + b0 + u) * Cout + c] = a;
    }
}

// se_fc_kernel: mean = b2 + (1/N) * sum of the K-slice partials (in slice order); scale = sigmoid(W2 relu(W1 mean))
// (sidekit/nnet/res_net.py:272-281).  One CTA per utterance; re-zeroes the fixed-point channel sums for the next block.
__global__ void __launch_bounds__(256) se_fc_kernel(unsigned long long* __restrict__ sums, const float* __restrict__ partial, int n_slices,
                                                    const int* __restrict__ utt_count, int B, int Cin, int Cout,
                                                    const float* __restrict__ b2, const float* __restrict__ fc1 /*[Cout/16][Cout]*/,
                                                    const float* __restrict__ fc2 /*[Cout][Cout/16]*/, float* __restrict__ scale) {
    __shared__ float mean[256];
    __shared__ float hid[16];
    pdl_wait();
    const int b = blockIdx.x;
    const float inv_n = 1.f / (float)utt_count[b];
    for (int c = threadIdx.x; c < Cin; c += blockDim.x) sums[(size_t)b * Cin + c] = 0ull;
    for (int co = threadIdx.x; co < Cout; co += blockDim.x) {
        float a = 0.f;
        for (int k = 0; k < n_slices; ++k) a += partial[((size_t)k * B + b) * Cout + co];
        mean[co] = fmaf(a, inv_n, b2[co]);
    }
    __syncthreads();
    const int R = Cout / 16;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (int jj = warp; jj < R; jj += blockDim.x >> 5) {
        float a = 0.f;
        for (int c = lane; c < Cout; c += 32) a = fmaf(fc1[jj * Cout + c], mean[c], a);
        a = warp_sum(a);
        if (lane == 0) hid[jj] = fmaxf(a, 0.f);
    }
    __syncthreads();
    for (int c = threadIdx.x; c < Cout; c += blockDim.x) {
        float a = 0.f;
        for (int jj = 0; jj < R; ++jj) a = fmaf(fc2[c * R + jj], hid[jj], a);
        scale[(size_t)b * Cout + c] = 1.f / (1.f + __expf(-a));
    }
}

int launch_se_scale(bool bf16, unsigned long long* sums, const uint16_t* y1, long long plane, int G, int Wp, int W,
                    const int* utt_row0, const int* utt_count, int B, int Cin, int Cout, const float* w2t, const float* b2,
                    const float* fc1, const float* fc2, float* brd_ws, float* scale, cudaStream_t st, const PlaneSumArgs* totals) {
    // brd_ws: [B][8][Cin] border sums, followed by [n_slices][B][Cout] partial means
    if (Cout > 256 || 256 % Cout != 0) {
        set_last_error(__FILE__, __LINE__, "squeeze-excitation: channel count must divide 256");
        return SKB_ERR_ARG;
    }
    dim3 grid(B, Cin / 8);
    SKB_CUDA_CHECK(launch_kernel(true, bf16 ? se_border_kernel<true> : se_border_kernel<false>, grid, dim3(256), 0, st, y1, plane, G, Wp, W, utt_row0,
                                 utt_count, Cin, brd_ws));
    // the channel totals (when conv1's epilogue did not produce them) run BESIDE the border sums: see plane_sum_kernel
    if (totals) {
        int rc = launch_plane_sum(bf16, y1, plane, G, totals->p_end, totals->pix_b, totals->span_b, Cin, sums, st);
        if (rc) return rc;
    }
    const int n_slices = Cin / kSeCh;
    float* partial = brd_ws + (size_t)B * 8 * Cin;
    dim3 g2(n_slices, (B + kSeUtt - 1) / kSeUtt);
    const auto mean_partial = Cout == 32 ? se_mean_partial_kernel<32> : Cout == 64 ? se_mean_partial_kernel<64>
                            : Cout == 128 ? se_mean_partial_kernel<128> : Cout == 256 ? se_mean_partial_kernel<256> : nullptr;
    if (!mean_partial) {
        set_last_error(__FILE__, __LINE__, "squeeze-excitation: unsupported channel count");
        return SKB_ERR_ARG;
    }
    SKB_CUDA_CHECK(launch_kernel(true, mean_partial, g2, dim3(256), 0, st, sums, brd_ws, B, Cin, w2t, partial));
    SKB_CUDA_CHECK(launch_kernel(true, se_fc_kernel, dim3(B), dim3(256), 0, st, sums, partial, n_slices, utt_count, B, Cin, Cout, b2, fc1, fc2, scale));
    return SKB_OK;
}

// ----------------------------------------------------------------------------- planes -> dense 16-bit frames
// X[frame][c * W + f] = act[c/8][G + (row0_b + t) * Wp + f][c%8]: the (B, C*F, T) view of
// sidekit/nnet/pooling.py:160-163, stored frame-major.  Thread per (frame, f, chunk).  The values stay in the 16-bit
// format of the activations (the statistics kernels widen them on the fly, which is exact): half the bytes of the
// former fp32 copy on the gather's write and on both readers.
template <bool BF16>
__global__ void gather_frames_kernel(const uint16_t* __restrict__ act, long long plane, int C, int W, int Wp, int G,
                                     const int* __restrict__ frame_row, int n_frames, uint16_t* __restrict__ X) {
    const int chunks = C >> 3;
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long total = (long long)n_frames * W * chunks;
    if (idx >= total) return;
    const int f = (int)(idx % W);
    const int j = (int)((idx / W) % chunks);
    const int fr = (int)(idx / ((long long)W * chunks));
    const long long pix = (long long)G + (long long)frame_row[fr] * Wp + f;
    const uint4 a = *reinterpret_cast<const uint4*>(act + ((size_t)j * plane + pix) * 8);
    const uint32_t u[4] = {a.x, a.y, a.z, a.w};
    uint16_t* dst = X + (size_t)fr * C * W;
#pragma unroll
    for (int e = 0; e < 4; ++e) {
        dst[(j * 8 + 2 * e) * W + f] = (uint16_t)(u[e] & 0xffffu);
        dst[(j * 8 + 2 * e + 1) * W + f] = (uint16_t)(u[e] >> 16);
    }
}

// The same gather as a packed tcgen05 operand (scoring.cu layout [frame / 128][chunk][frame % 128][8] halves) with the
// K index PERMUTED to k' = f * C + c: eight consecutive k' are eight consecutive channels of one pixel, i.e. exactly
// one 16-byte unit of the activation planes, so the operand is a straight copy (the weight matrix is packed with the
// same permutation).  The activations are 16-bit already: hi = the value, lo = 0 (the lo planes are zeroed once).
__global__ void gather_pack_kernel(const uint16_t* __restrict__ act, long long plane, int C, int W, int Wp, int G,
                                   const int* __restrict__ frame_row, int n_frames, uint16_t* __restrict__ hi) {
    const int chunks = C >> 3;                       // per f
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long total = (long long)n_frames * W * chunks;
    if (idx >= total) return;
    const int fr = (int)(idx % n_frames);            // consecutive threads = consecutive frames: contiguous 16-byte stores
    const int kc = (int)(idx / n_frames);            // chunk of k': f * chunks + j
    const int f = kc / chunks, j = kc - f * chunks;
    const long long pix = (long long)G + (long long)frame_row[fr] * Wp + f;
    const uint4 a = *reinterpret_cast<const uint4*>(act + ((size_t)j * plane + pix) * 8);
    const size_t o = (((size_t)(fr >> 7) * (W * chunks) + kc) * 128 + (fr & 127)) * 8;
    *reinterpret_cast<uint4*>(hi + o) = a;
}

int launch_gather_pack(const uint16_t* act, long long plane, int C, int W, int Wp, int G, const int* frame_row, int n_frames,
                       uint16_t* hi, cudaStream_t st) {
    const long long total = (long long)n_frames * W * (C / 8);
    if (total == 0) return SKB_OK;
    SKB_CUDA_CHECK(launch_kernel(false, gather_pack_kernel, (unsigned)((total + 255) / 256), 256, 0, st, act, plane, C, W, Wp, G, frame_row, n_frames,
                                 hi));
    return SKB_OK;
}

int launch_gather_frames(bool bf16, const uint16_t* act, long long plane, int C, int W, int Wp, int G,
                         const int* frame_row, int n_frames, uint16_t* X, cudaStream_t st) {
    const long long total = (long long)n_frames * W * (C / 8);
    const int threads = 256;
    const int blocks = (int)((total + threads - 1) / threads);
    if (blocks == 0) return SKB_OK;
    SKB_CUDA_CHECK(launch_kernel(false, bf16 ? gather_frames_kernel<true> : gather_frames_kernel<false>, blocks, threads, 0, st, act, plane, C, W, Wp,
                                 G, frame_row, n_frames, X));
    return SKB_OK;
}

// ----------------------------------------------------------------------------- mean / unbiased std over time
// MeanStdPooling (sidekit/nnet/pooling.py:55-70): out[b] = [mean_t x ; std_t x (ddof=1)].  Optional per-channel
// affine (s, t) applied as mean' = s*mean + t, std' = |s|*std (folds the TDNN's last BatchNorm).
// One CTA = 64 consecutive features (two per thread) x 8 time slices (threadIdx.y); a single pass with double accumulators (sum, sum of
// squares), the slices combined in slice order: deterministic, and in double as exact as the two-pass formula.
template <bool BF16>
__global__ void __launch_bounds__(256) meanstd_kernel(const uint16_t* __restrict__ X, const long long* __restrict__ frame_off,
                                                      const int* __restrict__ n_fr, int D, const float* __restrict__ aff_s,
                                                      const float* __restrict__ aff_t, float* __restrict__ out) {
    // a thread owns TWO consecutive features (one 32-bit load per frame: a warp reads 128 contiguous bytes); D is even
    __shared__ double ps[8][64], pss[8][64];
    const int b = blockIdx.y;
    const int d = (blockIdx.x * 32 + threadIdx.x) * 2;
    const int T = n_fr[b];
    double s[2] = {0.0, 0.0}, ss[2] = {0.0, 0.0};
    if (d < D) {
        const uint16_t* x = X + (size_t)frame_off[b] * D + d;
        for (int t = threadIdx.y; t < T; t += 8) {
            const float2 v2 = unpack2<BF16>(*reinterpret_cast<const uint32_t*>(x + (size_t)t * D));
            const double v0 = (double)v2.x, v1 = (double)v2.y;
            s[0] += v0; ss[0] = fma(v0, v0, ss[0]);
            s[1] += v1; ss[1] = fma(v1, v1, ss[1]);
        }
    }
#pragma unroll
    for (int q = 0; q < 2; ++q) {
        ps[threadIdx.y][2 * threadIdx.x + q] = s[q];
        pss[threadIdx.y][2 * threadIdx.x + q] = ss[q];
    }
    __syncthreads();
    if (threadIdx.y != 0 || d >= D) return;
#pragma unroll
    for (int q = 0; q < 2; ++q) {
        double a = 0.0, aa = 0.0;
        for (int k = 0; k < 8; ++k) { a += ps[k][2 * threadIdx.x + q]; aa += pss[k][2 * threadIdx.x + q]; }
        const double mean = a / T;
        const double var = fmax(aa - a * mean, 0.0) / (double)(T - 1);           // unbiased; T == 1 -> NaN like torch.std
        float sd = (float)sqrt(var);
        float mu = (float)mean;
        if (aff_s) {
            mu = aff_s[d + q] * mu + aff_t[d + q];
            sd = fabsf(aff_s[d + q]) * sd;
        }
        out[(size_t)b * 2 * D + d + q] = mu;
        out[(size_t)b * 2 * D + D + d + q] = sd;
    }
}

// MeanStdPooling straight from the 16-bit chunk planes of a W == 1 (TDNN) activation: one CTA per (utterance, 8-channel
// chunk); threads stride over the frames (16 contiguous bytes each, so a warp reads 512 contiguous bytes), double
// accumulators, fixed-order block reduction.  Replaces the fp32 gather (an uncoalesced 1.6 GB round trip on the
// 512-utterance TDNN batch) + the pooling pass over it.
template <bool BF16>
__global__ void __launch_bounds__(256) meanstd_planes_kernel(const uint16_t* __restrict__ act, long long plane, int G,
                                                             const int* __restrict__ utt_row0, const int* __restrict__ n_fr, int D,
                                                             const float* __restrict__ aff_s, const float* __restrict__ aff_t,
                                                             float* __restrict__ out) {
    // one WARP per (utterance, 8-channel chunk): lanes stride over the frames, shuffle reduction, no block barrier
    const int lane = threadIdx.x & 31;
    const int b = blockIdx.y, j = blockIdx.x * 8 + (threadIdx.x >> 5);
    if (j * 8 >= D) return;
    const int T = n_fr[b];
    const uint16_t* base = act + ((size_t)j * plane + G + utt_row0[b]) * 8;
    double s[8], ss[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) { s[e] = 0.0; ss[e] = 0.0; }
    for (int t0 = lane; t0 < T; t0 += 128) {
        uint4 a[4];                                        // four frames in flight per lane
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int t = t0 + 32 * u;
            a[u] = make_uint4(0u, 0u, 0u, 0u);             // zeros add nothing to either sum
            if (t < T) a[u] = *reinterpret_cast<const uint4*>(base + (size_t)t * 8);
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const uint32_t w[4] = {a[u].x, a[u].y, a[u].z, a[u].w};
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const float2 v = unpack2<BF16>(w[e]);
                s[2 * e] += (double)v.x; ss[2 * e] = fma((double)v.x, (double)v.x, ss[2 * e]);
                s[2 * e + 1] += (double)v.y; ss[2 * e + 1] = fma((double)v.y, (double)v.y, ss[2 * e + 1]);
            }
        }
    }
    double a_mine = 0.0, aa_mine = 0.0;
#pragma unroll
    for (int e = 0; e < 8; ++e) {
        for (int o = 16; o > 0; o >>= 1) {
            s[e] += __shfl_xor_sync(0xffffffffu, s[e], o);
            ss[e] += __shfl_xor_sync(0xffffffffu, ss[e], o);
        }
        if (lane == e) { a_mine = s[e]; aa_mine = ss[e]; }
    }
    if (lane < 8) {
        const int d = j * 8 + lane;
        const double mean = a_mine / T;
        const double var = fmax(aa_mine - a_mine * mean, 0.0) / (double)(T - 1);
        float mu = (float)mean, sd = (float)sqrt(var);
        if (aff_s) {
            mu = aff_s[d] * mu + aff_t[d];
            sd = fabsf(aff_s[d]) * sd;
        }
        out[(size_t)b * 2 * D + d] = mu;
        out[(size_t)b * 2 * D + D + d] = sd;
    }
}

int launch_meanstd_planes(bool bf16, const uint16_t* act, long long plane, int G, const int* utt_row0, const int* n_fr, int B, int D,
                          const float* aff_s, const float* aff_t, float* out, cudaStream_t st) {
    dim3 grid((D / 8 + 7) / 8, B);
    SKB_CUDA_CHECK(launch_kernel(false, bf16 ? meanstd_planes_kernel<true> : meanstd_planes_kernel<false>, grid, 256, 0, st, act, plane, G, utt_row0,
                                 n_fr, D, aff_s, aff_t, out));
    return SKB_OK;
}

int launch_meanstd(bool bf16, const uint16_t* X, const long long* frame_off, const int* n_fr, int B, int D, const float* aff_s,
                   const float* aff_t, float* out, cudaStream_t st) {
    if (D % 2 != 0) {
        set_last_error(__FILE__, __LINE__, "meanstd: the feature count must be even");
        return SKB_ERR_ARG;
    }
    dim3 grid((D + 63) / 64, B);
    SKB_CUDA_CHECK(launch_kernel(false, bf16 ? meanstd_kernel<true> : meanstd_kernel<false>, grid, dim3(32, 8), 0, st, X, frame_off, n_fr, D, aff_s,
                                 aff_t, out));
    return SKB_OK;
}

// ----------------------------------------------------------------------------- attention activation
// h = tanh(BN(relu(h + hb[utt])))  (sidekit/nnet/pooling.py:134-139: Conv1d -> ReLU -> BatchNorm1d -> Tanh);
// hb is the time-constant global-context part of the first Conv1d (+ its bias), one row per utterance.
__global__ void att_act_kernel(float* __restrict__ h, const float* __restrict__ hb, const int* __restrict__ frame_utt,
                               const float* __restrict__ bn_s, const float* __restrict__ bn_t, int n_frames, int A) {
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (long long)n_frames * A) return;
    const int fr = (int)(idx / A), a = (int)(idx % A);
    // ReLU that lets a NaN through like torch's does (fmaxf would turn it into 0): an utterance with a single pooled frame
    // has a NaN global-context std in the reference (unbiased estimator, pooling.py:68) and so a NaN embedding
    const float x = h[idx] + hb[(size_t)frame_utt[fr] * A + a];
    const float v = x > 0.f ? x : (x == x ? 0.f : x);
    h[idx] = tanhf(fmaf(v, bn_s[a], bn_t[a]));
}

int launch_att_act(float* h, const float* hb, const int* frame_utt, const float* bn_s, const float* bn_t, int n_frames,
                   int A, cudaStream_t st) {
    const long long total = (long long)n_frames * A;
    if (total == 0) return SKB_OK;
    SKB_CUDA_CHECK(launch_kernel(false, att_act_kernel, (int)((total + 255) / 256), 256, 0, st, h, hb, frame_utt, bn_s, bn_t, n_frames, A));
    return SKB_OK;
}

// ----------------------------------------------------------------------------- softmax over time + weighted stats
// w = softmax_t(logits); mu = sum x w; rh = sqrt(clamp(sum x^2 w - mu^2, 1e-9))  (pooling.py:167-169).
// One CTA = 32 consecutive features x 8 time slices; each slice runs an ONLINE softmax (running max with rescaling) over
// its frames in one pass over X and the logits, and the eight (max, sum e, sum x e, sum x^2 e) partials are merged in
// slice order.
template <bool BF16>
__global__ void __launch_bounds__(256) softmax_pool_kernel(const uint16_t* __restrict__ X, const float* __restrict__ logit,
                                                           const long long* __restrict__ frame_off, const int* __restrict__ n_fr, int D,
                                                           float* __restrict__ out) {
    // a thread owns TWO consecutive features: one 32-bit load of X and one 64-bit load of the logits per frame (D is even)
    __shared__ float pm[8][64], pe[8][64], px[8][64], pxx[8][64];
    const int b = blockIdx.y;
    const int d = (blockIdx.x * 32 + threadIdx.x) * 2;
    const int T = n_fr[b];
    float m[2] = {-INFINITY, -INFINITY}, se[2] = {0.f, 0.f}, sx[2] = {0.f, 0.f}, sxx[2] = {0.f, 0.f};
    if (d < D) {
        const size_t base = (size_t)frame_off[b] * D + d;
        for (int t0 = threadIdx.y; t0 < T; t0 += 32) {
            float2 lv[4], xv[4];                           // four frames' loads in flight before the dependent updates
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int t = t0 + 8 * u;
                lv[u] = t < T ? *reinterpret_cast<const float2*>(logit + base + (size_t)t * D) : make_float2(-INFINITY, -INFINITY);
                xv[u] = t < T ? unpack2<BF16>(*reinterpret_cast<const uint32_t*>(X + base + (size_t)t * D)) : make_float2(0.f, 0.f);
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                if (t0 + 8 * u >= T) break;
                const float lq[2] = {lv[u].x, lv[u].y}, xq[2] = {xv[u].x, xv[u].y};
#pragma unroll
                for (int q = 0; q < 2; ++q) {
                    const float l = lq[q], x = xq[q];
                    if (l > m[q]) {                        // new running max: rescale what has been accumulated
                        const float r = __expf(m[q] - l);  // exp(-inf) = 0 on the first frame
                        se[q] *= r; sx[q] *= r; sxx[q] *= r;
                        m[q] = l;
                    }
                    const float e = __expf(l - m[q]);
                    se[q] += e;
                    sx[q] = fmaf(x, e, sx[q]);
                    sxx[q] = fmaf(x * x, e, sxx[q]);
                }
            }
        }
    }
#pragma unroll
    for (int q = 0; q < 2; ++q) {
        const int c = 2 * threadIdx.x + q;
        pm[threadIdx.y][c] = m[q]; pe[threadIdx.y][c] = se[q];
        px[threadIdx.y][c] = sx[q]; pxx[threadIdx.y][c] = sxx[q];
    }
    __syncthreads();
    if (threadIdx.y != 0 || d >= D) return;
#pragma unroll
    for (int q = 0; q < 2; ++q) {
        const int c = 2 * threadIdx.x + q;
        float gm = -INFINITY;
        for (int k = 0; k < 8; ++k) gm = fmaxf(gm, pm[k][c]);
        float a = 0.f, ax = 0.f, axx = 0.f;
        for (int k = 0; k < 8; ++k) {
            const float r = __expf(pm[k][c] - gm);         // empty slices (T < 8): exp(-inf) = 0
            a = fmaf(pe[k][c], r, a);
            ax = fmaf(px[k][c], r, ax);
            axx = fmaf(pxx[k][c], r, axx);
        }
        const float mu = ax / a;
        const float var = axx / a - mu * mu;
        out[(size_t)b * 2 * D + d + q] = mu;
        out[(size_t)b * 2 * D + D + d + q] = sqrtf(fmaxf(var, 1e-9f));
    }
}

int launch_softmax_pool(bool bf16, const uint16_t* X, const float* logit, const long long* frame_off, const int* n_fr, int B, int D,
                        float* out, cudaStream_t st) {
    if (D % 2 != 0) {
        set_last_error(__FILE__, __LINE__, "softmax_pool: the feature count must be even");
        return SKB_ERR_ARG;
    }
    dim3 grid((D + 63) / 64, B);
    SKB_CUDA_CHECK(launch_kernel(false, bf16 ? softmax_pool_kernel<true> : softmax_pool_kernel<false>, grid, dim3(32, 8), 0, st, X, logit, frame_off,
                                 n_fr, D, out));
    return SKB_OK;
}

// ----------------------------------------------------------------------------- embedding head tail
// x -> optional per-feature affine (folded BatchNorm1d) -> l2_norm (loss.py:91-100, no eps)
// -> F.normalize (eps 1e-12) (xvector.py:893-903).  emb_pre = after l2_norm (input of the margin head),
// emb = the returned embedding.
__global__ void head_norm_kernel(const float* __restrict__ x, const float* __restrict__ aff_s, const float* __restrict__ aff_t,
                                 int E, int norm_embedding, float* __restrict__ emb_pre, float* __restrict__ emb) {
    extern __shared__ float hs[];
    __shared__ float red[32];
    const int b = blockIdx.x;
    float ss = 0.f;
    for (int i = threadIdx.x; i < E; i += blockDim.x) {
        float v = x[(size_t)b * E + i];
        if (aff_s) v = fmaf(v, aff_s[i], aff_t[i]);
        hs[i] = v;
        ss = fmaf(v, v, ss);
    }
    ss = warp_sum(ss);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = ss;
    __syncthreads();
    if (threadIdx.x < 32) {
        float v = threadIdx.x < (blockDim.x >> 5) ? red[threadIdx.x] : 0.f;
        v = warp_sum(v);
        if (threadIdx.x == 0) red[0] = v;
    }
    __syncthreads();
    const float nrm = sqrtf(red[0]);
    // l2_norm divides by the norm (no eps); F.normalize then divides by max(norm', 1e-12)
    const float s1 = norm_embedding ? 1.f / nrm : 1.f;
    const float n2 = norm_embedding ? (nrm * s1) : nrm;       // norm after the first step (== 1 up to rounding)
    const float s2 = 1.f / fmaxf(n2, 1e-12f);
    for (int i = threadIdx.x; i < E; i += blockDim.x) {
        const float v = hs[i] * s1;
        emb_pre[(size_t)b * E + i] = v;
        emb[(size_t)b * E + i] = v * s2;
    }
}

int launch_head_norm(const float* x, const float* aff_s, const float* aff_t, int B, int E, int norm_embedding,
                     float* emb_pre, float* emb, cudaStream_t st) {
    SKB_CUDA_CHECK(launch_kernel(false, head_norm_kernel, B, 256, E * sizeof(float), st, x, aff_s, aff_t, E, norm_embedding, emb_pre, emb));
    return SKB_OK;
}

// ----------------------------------------------------------------------------- fp32 SIMT GEMM (NT)
// C[m][n] = alpha * sum_k A[m][k] * B[n][k] + bias[n];  64x64 tile, 16-deep K slices, 4x4 register micro-tiles.
// Used for the small dense layers (attention projections, embedding and margin heads), which are
// < 0.5 % of the network's FLOPs and need fp32 inputs for the softmax logits.
// With gridDim.z > 1 the K range is split into slices of `k_slice` and slice z writes its partial tile to
// C + z * M * ldc (no bias / alpha): splitk_reduce_kernel adds the slices in order.
__global__ void __launch_bounds__(256) sgemm_nt_kernel(const float* __restrict__ A, const float* __restrict__ B,
                                                       float* __restrict__ C, const float* __restrict__ bias, int M, int N,
                                                       int K, int lda, int ldb, int ldc, float alpha, int k_slice) {
    __shared__ float As[16][64 + 4];
    __shared__ float Bs[16][64 + 4];
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    const int m0 = blockIdx.y * 64, n0 = blockIdx.x * 64;
    float acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
    const int lr = threadIdx.x >> 2;          // 0..63 row of the tile
    const int lk = (threadIdx.x & 3) * 4;     // 0,4,8,12
    const int k_begin = blockIdx.z * k_slice;
    if (gridDim.z > 1) {
        K = min(K, k_begin + k_slice);
        C += (size_t)blockIdx.z * M * ldc;
        bias = nullptr;
        alpha = 1.f;
    }
    for (int k0 = k_begin; k0 < K; k0 += 16) {
        {
            const int m = m0 + lr, n = n0 + lr;
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const int k = k0 + lk + e;
                As[lk + e][lr] = (m < M && k < K) ? A[(size_t)m * lda + k] : 0.f;
                Bs[lk + e][lr] = (n < N && k < K) ? B[(size_t)n * ldb + k] : 0.f;
            }
        }
        __syncthreads();
#pragma unroll
        for (int k = 0; k < 16; ++k) {
            float a[4], b[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) a[i] = As[k][ty * 4 + i];
#pragma unroll
            for (int j = 0; j < 4; ++j) b[j] = Bs[k][tx * 4 + j];
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
        }
        __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int m = m0 + ty * 4 + i;
        if (m >= M) continue;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int n = n0 + tx * 4 + j;
            if (n < N) C[(size_t)m * ldc + n] = alpha * acc[i][j] + (bias ? bias[n] : 0.f);
        }
    }
}

int launch_sgemm_nt(const float* A, const float* B, float* C, const float* bias, int M, int N, int K, int lda, int ldb,
                    int ldc, float alpha, cudaStream_t st) {
    if (M == 0 || N == 0) return SKB_OK;
    dim3 grid((N + 63) / 64, (M + 63) / 64);
    SKB_CUDA_CHECK(launch_kernel(false, sgemm_nt_kernel, grid, 256, 0, st, A, B, C, bias, M, N, K, lda, ldb, ldc, alpha, K));
    return SKB_OK;
}

__global__ void splitk_reduce_kernel(const float* __restrict__ part, int n_slices, int M, int N, const float* __restrict__ bias,
                                     float alpha, float* __restrict__ C, int ldc) {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= M * N) return;
    const int m = idx / N, n = idx - m * N;
    float a = 0.f;
    for (int z = 0; z < n_slices; ++z) a += part[((size_t)z * M + m) * N + n];          // fixed order: deterministic
    C[(size_t)m * ldc + n] = alpha * a + (bias ? bias[n] : 0.f);
}

// Skinny dense layer C[m][n] = alpha * sum_k A[m][k] W[n][k] + bias[n] for M = batch size (<= a few hundred rows) and
// large K (the 5120-wide pooled statistics): exact fp32 FMAs, K split over enough CTAs to fill the GPU, ordered
// reduction.  `ws` needs n_slices * M * N floats (skinny_gemm_ws_floats).
// The K split depends on N and K only -- never on the batch size M -- so that a row's summation order, and with it every
// embedding bit, is the same whatever batch the utterance travels in.
static int skinny_slices(int M, int N, int K) {
    (void)M;
    const int tiles = (N + 63) / 64;
    int z = (2 * kNumSMs + tiles - 1) / tiles;
    const int max_z = (K + 63) / 64;
    return z < 1 ? 1 : (z > max_z ? max_z : z);
}
size_t skinny_gemm_ws_floats(int M, int N, int K) { return (size_t)skinny_slices(M, N, K) * M * N; }

int launch_skinny_gemm(const float* A, int M, int K, const float* W, int N, const float* bias, float alpha, float* C, int ldc,
                       float* ws, cudaStream_t st) {
    if (M == 0 || N == 0) return SKB_OK;
    const int z = skinny_slices(M, N, K);
    const int k_slice = ((K + z - 1) / z + 15) / 16 * 16;
    const int zz = (K + k_slice - 1) / k_slice;
    dim3 grid((N + 63) / 64, (M + 63) / 64, zz);
    if (zz == 1) {
        SKB_CUDA_CHECK(launch_kernel(false, sgemm_nt_kernel, grid, 256, 0, st, A, W, C, bias, M, N, K, K, K, ldc, alpha, K));
    } else {
        SKB_CUDA_CHECK(launch_kernel(false, sgemm_nt_kernel, grid, 256, 0, st, A, W, ws, nullptr, M, N, K, K, K, N, 1.f, k_slice));
        SKB_CUDA_CHECK(launch_kernel(false, splitk_reduce_kernel, (M * N + 255) / 256, 256, 0, st, ws, zz, M, N, bias, alpha, C, ldc));
    }
    return SKB_OK;
}

// ----------------------------------------------------------------------------- fp32 frame-major -> 16-bit chunk planes
// Used by the TDNN path: (frames, C) features -> act[c/8][G + frame][8] (Wp == 1 geometry), zero padded channels.
template <bool BF16>
__global__ void pack_frames_kernel(const float* __restrict__ X, int C_src, int C_dst, int n_rows, const int* __restrict__ row_src,
                                   const int* __restrict__ row_b, const float2* __restrict__ cmvn /* [B][C_src] (mean, rstd) or null */,
                                   uint16_t* __restrict__ out, long long plane, int G) {
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const int chunks = C_dst >> 3;
    if (idx >= (long long)n_rows * chunks) return;
    const int row = (int)(idx % n_rows), j = (int)(idx / n_rows);
    const int src = row_src[row];
    const int b = (cmvn != nullptr && src >= 0) ? row_b[row] : -1;
    float v[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) {
        const int c = j * 8 + e;
        v[e] = (src >= 0 && c < C_src) ? X[(size_t)src * C_src + c] : 0.f;
        if (b >= 0 && c < C_src) {                     // CMVN on the fly, same arithmetic as cmvn_apply_kernel
            const float2 ms = __ldg(cmvn + (size_t)b * C_src + c);
            v[e] = (v[e] - ms.x) * ms.y;
        }
    }
    uint4 o;
    o.x = pack2<BF16>(v[0], v[1]); o.y = pack2<BF16>(v[2], v[3]); o.z = pack2<BF16>(v[4], v[5]); o.w = pack2<BF16>(v[6], v[7]);
    *reinterpret_cast<uint4*>(out + ((size_t)j * plane + G + row) * 8) = o;
}

int launch_pack_frames(bool bf16, const float* X, int C_src, int C_dst, int n_rows, const int* row_src, const int* row_b,
                       const float2* cmvn, uint16_t* out, long long plane, int G, cudaStream_t st) {
    const long long total = (long long)n_rows * (C_dst / 8);
    if (total == 0) return SKB_OK;
    const int blocks = (int)((total + 255) / 256);
    SKB_CUDA_CHECK(launch_kernel(false, bf16 ? pack_frames_kernel<true> : pack_frames_kernel<false>, blocks, 256, 0, st, X, C_src, C_dst, n_rows,
                                 row_src, row_b, cmvn, out, plane, G));
    return SKB_OK;
}

}  // namespace skb
