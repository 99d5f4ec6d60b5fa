// Shift-GEMM convolution on tcgen05 (sm_100a), persistent and fully pipelined.
//
// Activations live in HBM in a "chunk-plane, padded-linear" layout:
//     act[chunk j = c/8][pixel p][8 channels]   (16 bytes per (j, p), 16-bit elements)
// where pixels enumerate every line of every utterance back to back with ONE zero pad column per
// line (w == W) and ONE zero pad line between utterances:  p = G + row * Wp + w,  Wp = W + 1.
// In that layout a 3x3 / stride-1 / pad-1 convolution is nine GEMMs whose A operands are the SAME
// pixel slab shifted by (r-1)*Wp + (s-1) rows, and a contiguous run of pixels of one chunk plane is
// exactly one column of 8x16-byte UMMA core matrices (K-major, no swizzle).  So the kernel
//   * pulls each slab (128*MT output pixels + halo, 32 input channels) with one 1-D bulk copy per
//     chunk plane (cp.async.bulk, no tensor map, every input byte read ~once),
//   * streams the folded-BN weights, pre-packed on the host into per-(tap, k-chunk) UMMA images,
//   * issues tcgen05.mma M=128 x N x K=16 from one thread, descriptors differing per tap only in
//     their start address, accumulating MT tiles in TMEM,
//   * and eight epilogue warps read TMEM with tcgen05.ld, add the bias, apply the activation / pad
//     mask, optionally subsample (stride-2 convs are computed at stride 1 and every other pixel
//     kept), optionally apply the squeeze-excitation tail of a BasicBlock (acc * scale[utt][c] + residual,
//     ReLU -- the scales are known BEFORE this conv runs, see se_scale_kernel), and store 16-byte
//     channel groups, fully coalesced across the warp.
// One CTA per SM walks the (pixel tile, N split) work items round-robin.  Three mbarrier pipelines
// keep the roles decoupled across item boundaries: an A-slab ring and a weight ring (producers run
// ahead into the next items) and a double-buffered TMEM accumulator (the epilogue of item i overlaps
// the MMAs of item i+1).
// Replaces cuDNN conv + BN + ReLU kernels behind sidekit/nnet/res_net.py:309-320 and the Conv1d
// GEMMs of sidekit/nnet/xvector.py:467-483.
#pragma once
#include "common.cuh"

namespace skb {

struct ConvParams {
    const uint16_t* in;     // input planes
    long long in_plane;     // pixels per input chunk plane
    const uint16_t* w;      // packed weights: [n_split][kc][tap] images of [4][N_CTA][8]
    const uint16_t* w3;     // or nullptr: fused-tap packing [kc][r] images of [4][3 * Cout][8] (conv3_umma.cuh)
    int Wp;                 // pixels per padded line (fused-tap kernel)
    int n_utt;              // utterances in the batch (rows of se_scale)
    int scale_smem_bytes;   // fused-tap kernel: bytes of se_scale cached in shared memory (0 = read it from global memory)
    const float* bias;      // [cout] folded BN bias (fp32)
    uint16_t* out;          // output planes
    long long out_plane;
    int cin, cout, taps;    // taps = length of tap_shift[]
    // Tap groups: k-chunk kc belongs to group kc / kc_per_grp and uses taps [grp_tap[g], grp_tap[g+1]).  Ordinary convs have
    // one group with every tap.  A stride-2 conv reads a phase-split (space-to-depth) input: four phase images stacked as
    // channel chunks, each seen by its own subset of the nine taps (1 + 2 + 2 + 4).
    int kc_per_grp;
    int grp_tap[5];
    int n_pairs;            // (k-chunk, tap) pairs per work item = number of weight images per N split
    int G;                  // first computed pixel
    int p_end;              // one past the last computed pixel
    int halo;               // slab rows before the tile's first pixel (Wp + 1 for 3x3, 0 for 1x1 / causal taps)
    int rows_pad;           // slab rows per chunk plane (multiple of 8)
    int a_stages;           // slabs in the A ring (2..8)
    int b_stages;           // stages in the weight ring (2..8)
    int tps;                // taps per weight stage (divides taps): small layers fetch all taps of a k-chunk at once
    int b_resident;         // 1: all weight images of one N split fit in shared memory and are loaded once per CTA
    int n_tiles;            // pixel tiles
    int tap_shift[10];      // pixel shift of each tap: (r-1)*Wp + (s-1) for 3x3; k*dilation for the TDNN
    float act_slope;        // activation as max(x, slope * x): 1 = identity, 0 = ReLU, 0.2 = LeakyReLU(0.2)
    const int* pix_b;       // [p_end - G] utterance of each computed pixel, -1 for pad / invalid pixels
    const int* pix_sub;     // stride-2 convs: [p_end - G] destination pixel at the next level (even h, even w) or -1;
                            // nullptr for stride 1 (output pixel == input pixel)
    int bias_mma;           // 1: the bias is added by one extra MMA (ones x [bias_hi, bias_lo]) instead of the epilogue
    // fused squeeze-excitation tail (conv2 of a BasicBlock): out = act(acc * se_scale[b][n] + res[p][n])
    const float* se_scale;         // [B][cout] or nullptr
    const uint16_t* res;           // residual planes in the INPUT pixel geometry (block input or shortcut conv), or nullptr
    long long res_plane;
    // Per-(utterance, channel) totals of the STORED 16-bit outputs in 2^-15 fixed point (what plane_sum_kernel computes with
    // one more pass over the tensor), accumulated by the epilogue of an unfused, stride-1-output conv: [n_utt][cout] or
    // nullptr.  N_CTA == 32 with cout == 32: 32 per-thread 64-bit accumulators; N_CTA == 64 with cout == 64 and N_CTA == 128
    // with cout <= 256: the transposed ownership of ConvTotals.  Flushed with atomics when the utterance changes.
    unsigned long long* sums;
    unsigned* overflow;     // fp16 range guard: number of threads that stored a saturated (|x| >= 65504) value, or nullptr
    // Folded 1x1 shortcut (conv2 of a widening / striding block, N_CTA <= 64): the residual is computed here instead of read
    // from `res`.  Its input (the block input, or phase (0, 0) of a phase-split input: the first sc_cin / 8 planes) arrives
    // as extra halo-free k-chunks at the end of each item and accumulates into a second TMEM accumulator with the same
    // bias MMA and k-chunk order as a stand-alone 1x1 launch; the epilogue rounds it to 16 bits as that launch would store it.
    const uint16_t* sc_in;  // shortcut input planes (plane stride in_plane), or nullptr
    const uint16_t* sc_w;   // packed 1x1 weights: [n_split][sc_cin / 32] images of [4][N_CTA][8]
    const float* sc_bias;   // [cout] folded BN bias of the shortcut
    int sc_cin;
};

constexpr int kConvKC = 32;            // input channels per A/B stage (two K=16 MMAs)
constexpr int kConvMaxAStages = 8;
constexpr int kConvBStages = 8;
constexpr int kConvThreads = 12 * 32;  // warps: 0 A-producer, 1 B-producer, 2-3 MMA issuers, 4..11 epilogue (2 per TMEM quadrant)
constexpr int kConvCtrlBytes = 1024;
constexpr int kConvSmemBudget = 225 * 1024;

template <int N_CTA, int MT, bool SC = false>
struct ConvCfg {
    static constexpr int kAccCols = N_CTA * MT;        // one accumulator set
    static constexpr int kTmemCols = (SC ? 4 : 2) * kAccCols;   // double-buffered (+ the shortcut's): 256 or 512 columns
    static_assert(kTmemCols <= 512, "accumulators exceed tensor memory");
    static constexpr int kBStageBytes = N_CTA * kConvKC * 2;
    static constexpr int kTileM = 128 * MT;
    // ctrl | bias fp32 [cout] | ones operand (2 planes x 128 rows x 16 B) | bias images (2 planes x cout rows x 16 B) |
    // SE scales | SC: shortcut bias images (as the bias images) + shortcut weights [cout][sc_cin] | totals tiles | B | A
    static constexpr int kOnesBytes = 2 * 128 * 16;
    // channel totals with transposed ownership (ConvTotals, the TOT kernels): 32-row x 16-channel tiles per epilogue warp,
    // two (alternating chunks, one warp barrier per chunk) on the latency-bound 64-column epilogue
    static constexpr int kTotalsTileBytes = 32 * 16 * 2;
    static constexpr int kTotalsTiles = N_CTA == 64 ? 2 : 1;
    __host__ __device__ static size_t sc_bytes(int cout, int sc_cin) { return SC ? (size_t)cout * 32 + (size_t)cout * sc_cin * 2 : 0; }
    __host__ __device__ static constexpr size_t totals_bytes(bool tot) { return tot ? (size_t)8 * kTotalsTiles * kTotalsTileBytes : 0; }
    static size_t fixed_bytes(int cout, int bias_mma, int b_stages, int tps, int scale_bytes = 0, int sc_cin = 0, bool tot = false) {
        return kConvCtrlBytes + (size_t)cout * 4 + kOnesBytes + (bias_mma ? (size_t)cout * 32 : 0) + scale_bytes +
               sc_bytes(cout, sc_cin) + totals_bytes(tot) + (size_t)b_stages * tps * kBStageBytes;
    }
};

// Per-(utterance, channel) totals of the stored outputs on the 64- to 256-channel layers (ConvParams::sums): the integers
// plane_sum_kernel adds (2^-15 fixed point), so the result is bit-identical to that pass whatever the tile order, grid, N
// split or packing.  One accumulator per channel and thread, as on the 32-channel layers, would take 64-256 int64 registers
// here (168 registers and spills at 64 channels: profiles/r01g_rejected_experiments.txt), so ownership is transposed per
// epilogue warp: after storing a 16-channel chunk of its 32-row block, the warp also writes the packed words to a 1 KB
// shared-memory tile and reads it back column-wise.  Lane l owns channel pair p = l & 7 of the chunk and rows 4i + (l >> 3),
// i < 8 (conflict-free with the half swap below), and adds them to int64 registers that persist across items: acc[sel][k]
// holds channels (sel * KC + k) * 16 + 2p, + 1.  They reach memory only when the utterance changes and at the end of the
// CTA's range: two 64-bit shuffle-adds over the four row groups, one atomic per channel.  A block whose valid rows belong to
// more than one utterance (a few per utterance and level) adds each utterance's rows with atomics directly.
// The conversion is plane_sum's __float2int_rn(x * 2^15) computed as bits(fma(x, 2^15, 1.5 * 2^23)) - bits(1.5 * 2^23): the
// FMA rounds x * 2^15 + 1.5 * 2^23 once, to nearest even, and while the result stays in [2^23, 2^24) (|x| < 128) its
// significand is that integer exactly.  A lane sums its eight rows in 32 bits (< 2^25) and widens once; a lane with any value
// outside that binade (|x| >= 128, inf, NaN) takes F2I and 64-bit adds for the chunk instead.  NBUF = 2: chunks alternate
// between two tiles, so the tile of chunk c is rewritten only after the barrier of chunk c + 1, which every lane reaches after
// its reads of chunk c.
template <bool BF16, int NSEL, int KC, int NBUF>
struct ConvTotals {
    static_assert(NBUF == 1 || NBUF == 2, "one or two tiles per warp");
    static constexpr float kMagic = 12582912.f;            // 1.5 * 2^23
    static constexpr uint32_t kMagicBits = 0x4B400000u;
    long long acc[NSEL][KC][2];
    int b;               // utterance acc belongs to (warp-uniform), -1 = none yet
    int row_b;           // utterance of this lane's row of the current block
    unsigned valid;      // rows of the current block that hold an output
    bool mixed;          // the current block straddles utterances

    __device__ __forceinline__ void init() {
        b = -1;
        mixed = false;
#pragma unroll
        for (int s = 0; s < NSEL; ++s)
#pragma unroll
            for (int k = 0; k < KC; ++k) acc[s][k][0] = acc[s][k][1] = 0ll;
    }
    __device__ __forceinline__ static void fix_add2(uint32_t w, long long& t0, long long& t1) {   // plane_sum_kernel's arithmetic
        float2 f = unpack2<BF16>(w);
        if (BF16) { f.x = fminf(fmaxf(f.x, -65504.f), 65504.f); f.y = fminf(fmaxf(f.y, -65504.f), 65504.f); }
        t0 += (long long)__float2int_rn(f.x * 32768.f);
        t1 += (long long)__float2int_rn(f.y * 32768.f);
    }
    __device__ __forceinline__ void flush(unsigned long long* sums, int cout, int lane) {
        if (b < 0) return;
#pragma unroll
        for (int s = 0; s < NSEL; ++s)
#pragma unroll
            for (int k = 0; k < KC; ++k)
#pragma unroll
                for (int e = 0; e < 2; ++e) {
                    long long v = acc[s][k][e];
                    v += shfl_xor_ll(v, 8);
                    v += shfl_xor_ll(v, 16);
                    if (lane < 8 && v != 0ll)
                        atomicAdd(sums + (size_t)b * cout + (s * KC + k) * 16 + 2 * lane + e, (unsigned long long)v);
                    acc[s][k][e] = 0ll;
                }
    }
    // once per 32-row block, by the whole warp, before its chunks: the fast path needs every valid row in utterance b
    __device__ __forceinline__ void begin_block(int bidx, unsigned long long* sums, int cout, int lane) {
        row_b = bidx;
        valid = __ballot_sync(0xffffffffu, bidx >= 0);
        mixed = false;
        const unsigned other = __ballot_sync(0xffffffffu, bidx >= 0 && bidx != b);
        if (other != 0u) {
            const int nb = __shfl_sync(0xffffffffu, bidx, __ffs(other) - 1);
            if (__ballot_sync(0xffffffffu, bidx >= 0 && bidx != nb) != 0u) {
                mixed = true;
            } else {
                flush(sums, cout, lane);
                b = nb;
            }
        }
    }
    // this lane's row (= lane) of the chunk, 16 channels as two packed uint4 (j = 0, 1), zeros for rows without output;
    // the 16-byte halves of every other group of four rows are swapped so that the column reads hit 32 distinct banks
    __device__ __forceinline__ static void put(uint4* tile, int lane, int j, const uint4& o) {
        tile[lane * 2 + (j ^ ((lane >> 2) & 1))] = o;
    }
    // after both put()s of a chunk, by the whole warp; sel is warp-uniform, k a compile-time constant after unrolling
    __device__ __forceinline__ void add_chunk(const uint4* tile, int sel, int k, unsigned long long* sums, int cout, int lane) {
        __syncwarp();
        const uint32_t* t = reinterpret_cast<const uint32_t*>(tile);
        const int p = lane & 7, rg = lane >> 3;
        uint32_t w[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) w[i] = t[(4 * i + rg) * 8 + ((((p >> 2) ^ (i & 1))) << 2) + (p & 3)];
        if (NBUF == 1) __syncwarp();         // the tile is free for the next chunk
        if (!mixed) {
            uint32_t all = 0xffffffffu, any = 0u, s0 = 0u, s1 = 0u;     // the sums wrap; their difference below does not
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const float2 f = unpack2<BF16>(w[i]);
                const uint32_t r0 = __float_as_uint(fmaf(f.x, 32768.f, kMagic)), r1 = __float_as_uint(fmaf(f.y, 32768.f, kMagic));
                all &= r0 & r1;
                any |= r0 | r1;
                s0 += r0;
                s1 += r1;
            }
            long long t0, t1;
            if ((all & 0xFF800000u) == 0x4B000000u && (any & 0xFF800000u) == 0x4B000000u) {   // every result in [2^23, 2^24)
                t0 = (long long)(int)(s0 - 8u * kMagicBits);
                t1 = (long long)(int)(s1 - 8u * kMagicBits);
            } else {
                t0 = t1 = 0ll;
#pragma unroll
                for (int i = 0; i < 8; ++i) fix_add2(w[i], t0, t1);
            }
#pragma unroll
            for (int s = 0; s < NSEL; ++s)
                if (s == sel) { acc[s][k][0] += t0; acc[s][k][1] += t1; }
            return;
        }
        unsigned left = valid;
        while (left != 0u) {
            const int u = __shfl_sync(0xffffffffu, row_b, __ffs(left) - 1);
            const unsigned m = __ballot_sync(0xffffffffu, row_b == u);
            left &= ~m;
            long long t0 = 0ll, t1 = 0ll;
#pragma unroll
            for (int i = 0; i < 8; ++i)
                if ((m >> (4 * i + rg)) & 1u) fix_add2(w[i], t0, t1);
            t0 += shfl_xor_ll(t0, 8); t0 += shfl_xor_ll(t0, 16);
            t1 += shfl_xor_ll(t1, 8); t1 += shfl_xor_ll(t1, 16);
            unsigned long long* dst = sums + (size_t)u * cout + (sel * KC + k) * 16 + 2 * p;
            if (lane < 8 && t0 != 0ll) atomicAdd(dst, (unsigned long long)t0);
            if (lane < 8 && t1 != 0ll) atomicAdd(dst + 1, (unsigned long long)t1);
        }
    }
};

// TOT: this instantiation accumulates ConvParams::sums (non-null) with ConvTotals; the others carry none of its code
template <int N_CTA, int MT, bool BF16, bool FUSED, bool SC = false, bool TOT = false>
__global__ void __launch_bounds__(kConvThreads, 1) conv_umma_kernel(const ConvParams p) {
    static_assert(!SC || (FUSED && N_CTA <= 64), "the folded shortcut exists for the narrow conv2 epilogue only");
    static_assert(!TOT || (!FUSED && N_CTA >= 64), "ConvTotals: the unfused 64- and 128-column epilogues");
    using Cfg = ConvCfg<N_CTA, MT, SC>;
    extern __shared__ __align__(128) uint8_t smem[];
    uint64_t* a_full = reinterpret_cast<uint64_t*>(smem);           // [kConvMaxAStages]
    uint64_t* a_empty = a_full + kConvMaxAStages;
    uint64_t* b_full = a_empty + kConvMaxAStages;                   // [kConvBStages]
    uint64_t* b_empty = b_full + kConvBStages;
    uint64_t* acc_full = b_empty + kConvBStages;                    // [2]
    uint64_t* acc_empty = acc_full + 2;                             // [2]
    uint64_t* sc_full = acc_empty + 2;                              // SC: shortcut weights resident
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(sc_full + 1);
    float* bias_s = reinterpret_cast<float*>(smem + kConvCtrlBytes);
    uint8_t* ones_smem = smem + kConvCtrlBytes + (size_t)p.cout * 4;
    uint8_t* biasimg_smem = ones_smem + Cfg::kOnesBytes;          // per N split: [2 planes][N_CTA rows][8 halves]
    float* scale_s = reinterpret_cast<float*>(biasimg_smem + (p.bias_mma ? (size_t)p.cout * 32 : 0));   // [n_utt][cout] SE scales
    uint8_t* sc_biasimg_smem = reinterpret_cast<uint8_t*>(scale_s) + p.scale_smem_bytes;
    uint8_t* sc_w_smem = sc_biasimg_smem + (size_t)p.cout * 32;
    uint8_t* totals_smem = reinterpret_cast<uint8_t*>(scale_s) + p.scale_smem_bytes + Cfg::sc_bytes(p.cout, p.sc_cin);   // ConvTotals tiles
    uint8_t* b_smem = totals_smem + Cfg::totals_bytes(TOT);
    const uint32_t b_stage_bytes = (uint32_t)p.tps * Cfg::kBStageBytes;
    uint8_t* a_smem = b_smem + (size_t)p.b_stages * b_stage_bytes;
    const uint32_t a_stage_bytes = (uint32_t)p.rows_pad * (kConvKC / 8) * 16;

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const int n_split = p.cout / N_CTA;
    const int n_items = p.n_tiles * n_split;
    const int n_kc = p.cin / kConvKC;
    // Every CTA walks a CONTIGUOUS range of work items (item = tile * n_split + N split): the N splits of a tile follow each
    // other on the same SM (the slab comes back from L2), and an epilogue thread stays inside one utterance for hundreds of
    // tiles.
    const int item_begin = (int)((long long)n_items * blockIdx.x / gridDim.x);
    const int item_end = (int)((long long)n_items * (blockIdx.x + 1) / gridDim.x);

    if (threadIdx.x == 0) {
        // two MMA-issuing warps (one half of the accumulator tiles each) arrive on the "consumed" barriers
        for (int i = 0; i < kConvMaxAStages; ++i) { mbar_init(&a_full[i], 1); mbar_init(&a_empty[i], 2); }
        for (int i = 0; i < kConvBStages; ++i) { mbar_init(&b_full[i], 1); mbar_init(&b_empty[i], 2); }   // first b_stages used
        for (int i = 0; i < 2; ++i) { mbar_init(&acc_full[i], 2); mbar_init(&acc_empty[i], 8); }
        if (SC) mbar_init(sc_full, 1);
        fence_barrier_init();
    }
    for (int i = threadIdx.x; i < p.cout; i += blockDim.x) bias_s[i] = p.bias[i];
    if (p.bias_mma) {
        // "ones" A operand: every row = (1, 1, 0, ..., 0) over K = 16; bias B operand: row n = (hi_n, lo_n, 0, ..., 0) with
        // hi + lo = bias to ~2^-22: one extra K=16 MMA per accumulator tile initialises it with the bias.
        const uint32_t one2 = pack2<BF16>(1.f, 1.f);
        for (int i = threadIdx.x; i < 2 * 128; i += blockDim.x)
            reinterpret_cast<uint4*>(ones_smem)[i] = make_uint4(i < 128 ? one2 : 0u, 0u, 0u, 0u);
        auto bias_images = [&](const float* bias, uint8_t* dst) {
            for (int i = threadIdx.x; i < 2 * p.cout; i += blockDim.x) {
                const int ns = (i % p.cout) / N_CTA, n = (i % p.cout) % N_CTA, plane = i / p.cout;
                uint32_t w0 = 0u;
                if (plane == 0) {
                    const float b = bias[ns * N_CTA + n];
                    const float2 hi2 = unpack2<BF16>(pack2<BF16>(b, 0.f));
                    w0 = pack2<BF16>(b, b - hi2.x);
                }
                reinterpret_cast<uint4*>(dst)[(size_t)ns * 2 * N_CTA + plane * N_CTA + n] = make_uint4(w0, 0u, 0u, 0u);
            }
        };
        bias_images(p.bias, biasimg_smem);
        if (SC) bias_images(p.sc_bias, sc_biasimg_smem);
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    if (warp == 2) tmem_alloc<Cfg::kTmemCols>(tmem_slot);
    // everything above touches only constants (weights, bias) and this CTA's shared / tensor memory: it overlaps the tail of
    // the previous kernel of the stream.  From here on the kernel reads what that kernel wrote.
    pdl_wait();
    if (FUSED && p.scale_smem_bytes > 0)
        for (int i = threadIdx.x; i < p.scale_smem_bytes / 4; i += blockDim.x) scale_s[i] = p.se_scale[i];
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        // ---------------------------------------------------------------- A producer: activation slabs
        if (lane == 0) {
            const uint32_t plane_bytes = (uint32_t)p.rows_pad * 16;
            int s = 0;
            uint32_t ph = 1;     // ring position / parity kept incrementally (no divisions on the critical paths)
            int tile = item_begin / n_split, ns_ctr = item_begin % n_split;
            for (int item = item_begin; item < item_end; ++item) {
                const long long q0 = (long long)p.G + (long long)tile * Cfg::kTileM - p.halo;   // >= 0 thanks to the guard G
                if (++ns_ctr == n_split) { ns_ctr = 0; ++tile; }
                for (int kc = 0; kc < n_kc; ++kc) {
                    mbar_wait(&a_empty[s], ph);
                    mbar_arrive_expect_tx(&a_full[s], a_stage_bytes);
#pragma unroll
                    for (int j = 0; j < kConvKC / 8; ++j) {
                        const uint16_t* src = p.in + ((size_t)(kc * (kConvKC / 8) + j) * p.in_plane + q0) * 8;
                        bulk_g2s(a_smem + (size_t)s * a_stage_bytes + j * plane_bytes, src, plane_bytes, &a_full[s]);
                    }
                    if (++s == p.a_stages) { s = 0; ph ^= 1; }
                }
                if constexpr (SC) {
                    // shortcut chunks: the tile's own pixels, no halo (same plane stride inside the stage as the slab)
                    constexpr uint32_t sc_plane_bytes = Cfg::kTileM * 16;
                    const long long qs = q0 + p.halo;
                    for (int kc = 0; kc < p.sc_cin / kConvKC; ++kc) {
                        mbar_wait(&a_empty[s], ph);
                        mbar_arrive_expect_tx(&a_full[s], (kConvKC / 8) * sc_plane_bytes);
#pragma unroll
                        for (int j = 0; j < kConvKC / 8; ++j) {
                            const uint16_t* src = p.sc_in + ((size_t)(kc * (kConvKC / 8) + j) * p.in_plane + qs) * 8;
                            bulk_g2s(a_smem + (size_t)s * a_stage_bytes + j * plane_bytes, src, sc_plane_bytes, &a_full[s]);
                        }
                        if (++s == p.a_stages) { s = 0; ph ^= 1; }
                    }
                }
            }
        }
    } else if (warp == 1) {
        // ---------------------------------------------------------------- B producer: packed weights
        if (lane == 0) {
            const int n_it = p.n_pairs;                // weight images per item
            if constexpr (SC) {
                const uint32_t bytes = (uint32_t)p.cout * p.sc_cin * 2;
                mbar_arrive_expect_tx(sc_full, bytes);
                bulk_g2s(sc_w_smem, p.sc_w, bytes, sc_full);
            }
            if (p.b_resident) {
                // small layers: the whole weight tensor stays in shared memory for the life of the CTA
                mbar_arrive_expect_tx(&b_full[0], (uint32_t)n_it * Cfg::kBStageBytes);
                for (int it = 0; it < n_it; ++it)
                    bulk_g2s(b_smem + (size_t)it * Cfg::kBStageBytes, p.w + (size_t)it * (Cfg::kBStageBytes / 2), Cfg::kBStageBytes,
                             &b_full[0]);
            } else {
                const int n_st = n_it / p.tps;             // weight stages per item
                int s = 0;
                uint32_t ph = 1;
                int ns = item_begin % n_split;
                for (int item = item_begin; item < item_end; ++item) {
                    const uint16_t* wbase = p.w + (size_t)ns * n_it * (Cfg::kBStageBytes / 2);
                    if (++ns == n_split) ns = 0;
                    for (int it = 0; it < n_st; ++it) {
                        mbar_wait(&b_empty[s], ph);
                        mbar_arrive_expect_tx(&b_full[s], b_stage_bytes);
                        bulk_g2s(b_smem + (size_t)s * b_stage_bytes, wbase + (size_t)it * (b_stage_bytes / 2), b_stage_bytes,
                                 &b_full[s]);
                        if (++s == p.b_stages) { s = 0; ph ^= 1; }
                    }
                }
            }
        }
    } else if (warp == 2 || warp == 3) {
        // ---------------------------------------------------------------- MMA issuers
        // Two warps, each owning half of the item's MT accumulator tiles (fixed per-accumulator MMA order, so the
        // result does not depend on their relative timing): issue bandwidth, not the tensor pipe, limits small-N MMAs.
        // The whole warp walks the loops (addresses / descriptors stay warp-uniform); one elected lane issues.
        constexpr int MTW = MT / 2;
        const int mtw0 = (warp - 2) * MTW;
        const uint32_t idesc = umma_idesc_f16(128, N_CTA, BF16);
        const uint32_t a_lbo = (uint32_t)p.rows_pad * 16;   // next 8-channel plane of the slab
        const uint32_t b_lbo = N_CTA * 16;
        const uint64_t desc_hi_a = (static_cast<uint64_t>((a_lbo >> 4) & 0x3FFF) << 16) | (static_cast<uint64_t>(128 >> 4) << 32) |
                                   (static_cast<uint64_t>(1) << 46);
        const uint64_t desc_hi_b = (static_cast<uint64_t>((b_lbo >> 4) & 0x3FFF) << 16) | (static_cast<uint64_t>(128 >> 4) << 32) |
                                   (static_cast<uint64_t>(1) << 46);
        int as = 0, bs = 0, ns = item_begin % n_split;
        uint32_t a_ph = 0, b_ph = 0, n_done = 0;
        if (p.b_resident) {
            mbar_wait(&b_full[0], 0);
            tc_fence_after();
        }
        if constexpr (SC) {
            mbar_wait(sc_full, 0);
            tc_fence_after();
        }
        const uint64_t ones_desc = (static_cast<uint64_t>(2048 >> 4) << 16) | (static_cast<uint64_t>(128 >> 4) << 32) |
                                   (static_cast<uint64_t>(1) << 46) | ((smem_u32(ones_smem) >> 4) & 0x3FFF);
        for (int item = item_begin; item < item_end; ++item, ++n_done) {
            const int buf = (int)(n_done & 1);
            mbar_wait(&acc_empty[buf], ((n_done >> 1) & 1) ^ 1);
            tc_fence_after();
            const uint32_t d_tmem = tmem_base + buf * Cfg::kAccCols;
            const int ns_item = ns;
            if (++ns == n_split) ns = 0;
            if (p.bias_mma && elect_one()) {
                const uint32_t img = smem_u32(biasimg_smem) + (uint32_t)ns_item * 2 * N_CTA * 16;
                const uint64_t bias_desc = desc_hi_b | ((img >> 4) & 0x3FFF);
#pragma unroll
                for (int mt = mtw0; mt < mtw0 + MTW; ++mt) umma_f16(d_tmem + mt * N_CTA, ones_desc, bias_desc, idesc, 0u);
            }
            __syncwarp();
            const uint32_t acc0 = p.bias_mma ? 1u : 0u;
            int grp = 0, in_grp = 0, flat = 0;
            bool first = true;                       // first MMA of the item overwrites (or follows the bias MMA)
            for (int kc = 0; kc < n_kc; ++kc) {
                mbar_wait(&a_full[as], a_ph);
                tc_fence_after();
                const uint32_t a_base = smem_u32(a_smem + (size_t)as * a_stage_bytes) + (uint32_t)p.halo * 16;
                const int tb = p.grp_tap[grp], te = p.grp_tap[grp + 1];
                const int tstep = p.b_resident ? (te - tb) : p.tps;
                for (int tap0 = tb; tap0 < te; tap0 += tstep) {
                    uint32_t b_stage;
                    if (p.b_resident) {
                        b_stage = smem_u32(b_smem) + (uint32_t)flat * Cfg::kBStageBytes;
                    } else {
                        mbar_wait(&b_full[bs], b_ph);
                        tc_fence_after();
                        b_stage = smem_u32(b_smem + (size_t)bs * b_stage_bytes);
                    }
                    if (elect_one()) {
                        for (int tt = 0; tt < tstep; ++tt) {
                            const int tap = tap0 + tt;
                            const uint32_t a_tap = a_base + (uint32_t)(p.tap_shift[tap] * 16);
                            const uint32_t b_tap = b_stage + tt * Cfg::kBStageBytes;
#pragma unroll
                            for (int ks = 0; ks < kConvKC / 16; ++ks) {
                                const uint64_t bdesc = desc_hi_b | (((b_tap + ks * 2 * b_lbo) >> 4) & 0x3FFF);
#pragma unroll
                                for (int mt = mtw0; mt < mtw0 + MTW; ++mt) {
                                    const uint64_t adesc = desc_hi_a | (((a_tap + ks * 2 * a_lbo + mt * 2048) >> 4) & 0x3FFF);
                                    umma_f16(d_tmem + mt * N_CTA, adesc, bdesc, idesc, (!first || tt > 0 || ks > 0) ? 1u : acc0);
                                }
                            }
                        }
                        if (!p.b_resident) umma_commit(&b_empty[bs]);
                    }
                    __syncwarp();
                    first = false;
                    flat += tstep;
                    if (!p.b_resident && ++bs == p.b_stages) { bs = 0; b_ph ^= 1; }
                }
                if (elect_one()) umma_commit(&a_empty[as]);
                __syncwarp();
                if (++as == p.a_stages) { as = 0; a_ph ^= 1; }
                if (++in_grp == p.kc_per_grp) { in_grp = 0; ++grp; }
            }
            if constexpr (SC) {
                // the shortcut's accumulator: bias MMA, then its k-chunks in order -- a stand-alone 1x1 launch's sequence
                const uint32_t dsc_tmem = tmem_base + (2 + buf) * Cfg::kAccCols;
                if (elect_one()) {
                    const uint32_t img = smem_u32(sc_biasimg_smem) + (uint32_t)ns_item * 2 * N_CTA * 16;
                    const uint64_t bias_desc = desc_hi_b | ((img >> 4) & 0x3FFF);
#pragma unroll
                    for (int mt = mtw0; mt < mtw0 + MTW; ++mt) umma_f16(dsc_tmem + mt * N_CTA, ones_desc, bias_desc, idesc, 0u);
                }
                __syncwarp();
                const int sc_kc = p.sc_cin / kConvKC;
                for (int kc = 0; kc < sc_kc; ++kc) {
                    mbar_wait(&a_full[as], a_ph);
                    tc_fence_after();
                    const uint32_t a_base = smem_u32(a_smem + (size_t)as * a_stage_bytes);
                    const uint32_t b_img = smem_u32(sc_w_smem) + (uint32_t)(ns_item * sc_kc + kc) * Cfg::kBStageBytes;
                    if (elect_one()) {
#pragma unroll
                        for (int ks = 0; ks < kConvKC / 16; ++ks) {
                            const uint64_t bdesc = desc_hi_b | (((b_img + ks * 2 * b_lbo) >> 4) & 0x3FFF);
#pragma unroll
                            for (int mt = mtw0; mt < mtw0 + MTW; ++mt) {
                                const uint64_t adesc = desc_hi_a | (((a_base + ks * 2 * a_lbo + mt * 2048) >> 4) & 0x3FFF);
                                umma_f16(dsc_tmem + mt * N_CTA, adesc, bdesc, idesc, 1u);
                            }
                        }
                        umma_commit(&a_empty[as]);
                    }
                    __syncwarp();
                    if (++as == p.a_stages) { as = 0; a_ph ^= 1; }
                }
            }
            if (elect_one()) umma_commit(&acc_full[buf]);
            __syncwarp();
        }
    } else if (warp >= 4) {
        if constexpr (N_CTA <= 64) {
        // ---------------------------------------------------------------- epilogue warps (4..11), narrow layers
        // Two warps per TMEM lane quadrant, each taking half of the item's MT accumulator tiles.  Per-pixel metadata
        // and the residual come from HBM / L2 (~1 us away) and depend on each other (pixel -> utterance -> residual
        // row / scale row); on these layers an item is only ~3 k cycles of MMAs, so that chain -- paid once per item --
        // was the critical path (profiles/r01c_fused_taps.txt).  Metadata is therefore fetched TWO items ahead, the
        // residual ONE item ahead, and the SE scale table sits in shared memory.
        constexpr int MTH = MT / 2;
        constexpr int NCH = N_CTA / 8;          // 8-channel chunks per pixel (4 or 8): the whole residual is one group
        const int q = warp & 3;                 // TMEM lane quadrant this warp may read
        const int mt0 = ((warp - 4) >> 2) * MTH;
        const size_t plane8 = (size_t)p.out_plane * 8;
        const size_t rplane8 = (size_t)p.res_plane * 8;
        const float slope = p.act_slope;
        auto fetch_meta = [&](int item, int (&bidx)[MTH], int (&opix)[MTH]) {
            const int tile = item / n_split;
#pragma unroll
            for (int mt = 0; mt < MTH; ++mt) {
                const int pix = p.G + tile * Cfg::kTileM + (mt0 + mt) * 128 + q * 32 + lane;
                const bool in_range = item < item_end && pix < p.p_end;
                bidx[mt] = in_range ? __ldg(p.pix_b + (pix - p.G)) : -1;
                opix[mt] = in_range ? pix : -1;
                if (p.pix_sub != nullptr) opix[mt] = in_range ? __ldg(p.pix_sub + (pix - p.G)) : -1;
            }
        };
        auto fetch_res = [&](int item, const int (&bidx)[MTH], uint4 (&rv)[MTH][NCH]) {
            const int tile = item / n_split, n_base = (item - tile * n_split) * N_CTA;
#pragma unroll
            for (int mt = 0; mt < MTH; ++mt) {
                const size_t roff = (size_t)(p.G + tile * Cfg::kTileM + (mt0 + mt) * 128 + q * 32 + lane) * 8;
#pragma unroll
                for (int k = 0; k < NCH; ++k) {
                    rv[mt][k] = make_uint4(0u, 0u, 0u, 0u);
                    if (bidx[mt] >= 0) rv[mt][k] = *reinterpret_cast<const uint4*>(p.res + roff + (size_t)((n_base >> 3) + k) * rplane8);
                }
            }
        };
        constexpr bool kLoadRes = FUSED && !SC;  // with SC the residual is the shortcut accumulator in TMEM
        uint32_t omax = 0u;                     // fp16 range guard: max |x| of what this thread stored
        int bidx_c[MTH], opix_c[MTH], bidx_n[MTH], opix_n[MTH], bidx_nn[MTH], opix_nn[MTH];
        uint4 rv_c[MTH][NCH], rv_n[MTH][NCH];
        fetch_meta(item_begin, bidx_c, opix_c);
        fetch_meta(item_begin + 1, bidx_n, opix_n);
        if (kLoadRes) fetch_res(item_begin, bidx_c, rv_c);
        uint32_t n_done = 0;
        // fused channel totals (see ConvParams::sums): this thread's pixels stay inside one utterance for hundreds of
        // consecutive tiles, so the totals live in registers and reach memory only when the utterance changes
        constexpr bool kCanSum = (N_CTA == 32) && !FUSED;
        constexpr int kSumRegs = kCanSum ? 32 : 1;
        long long sacc[kSumRegs];
        int sum_b = -1;
#pragma unroll
        for (int i = 0; i < kSumRegs; ++i) sacc[i] = 0ll;
        const bool do_sums = kCanSum && p.sums != nullptr;
        auto flush_sums = [&]() {
            if (sum_b >= 0) {
#pragma unroll
                for (int i = 0; i < kSumRegs; ++i) {
                    if (sacc[i] != 0ll) atomicAdd(p.sums + (size_t)sum_b * p.cout + i, (unsigned long long)sacc[i]);
                    sacc[i] = 0ll;
                }
            }
        };
        // 64 channels: transposed ownership (ConvTotals), one 32-row block per warp and item
        constexpr bool kTSum = TOT;
        static_assert(!kTSum || MTH == 1, "ConvTotals takes one 32-row block per warp and item");
        static_assert(!kTSum || (NCH / 2) % Cfg::kTotalsTiles == 0, "chunks per item: a multiple of the tiles (parity across items)");
        ConvTotals<BF16, 1, N_CTA / 16, Cfg::kTotalsTiles> tot;
        uint4* tot_tile = reinterpret_cast<uint4*>(totals_smem + (warp - 4) * Cfg::kTotalsTiles * Cfg::kTotalsTileBytes);
        if constexpr (kTSum) tot.init();
        for (int item = item_begin; item < item_end; ++item, ++n_done) {
            const int tile = item / n_split;
            const int n_base = (item - tile * n_split) * N_CTA;
            const int buf = (int)(n_done & 1);
            if (kLoadRes) fetch_res(item + 1, bidx_n, rv_n);               // its metadata arrived during the previous item
            fetch_meta(item + 2, bidx_nn, opix_nn);
            if constexpr (kTSum) tot.begin_block(bidx_c[0], p.sums, p.cout, lane);   // a flush overlaps the MMAs
            mbar_wait(&acc_full[buf], (n_done >> 1) & 1);
            tc_fence_after();
#pragma unroll
            for (int cc = 0; cc < NCH; cc += 2) {
                const int c0 = cc * 8;
#pragma unroll
                for (int mt = 0; mt < MTH; ++mt) {
                    const bool valid = bidx_c[mt] >= 0;
                    if (kCanSum && do_sums && valid && bidx_c[mt] != sum_b) {
                        flush_sums();
                        sum_b = bidx_c[mt];
                    }
                    float4 sc4[4];
                    if (FUSED && valid) {
                        if (p.scale_smem_bytes > 0) {
                            const float4* sp = reinterpret_cast<const float4*>(scale_s + (size_t)bidx_c[mt] * p.cout + n_base + c0);
#pragma unroll
                            for (int k = 0; k < 4; ++k) sc4[k] = sp[k];
                        } else {
                            const float4* sp = reinterpret_cast<const float4*>(p.se_scale + (size_t)bidx_c[mt] * p.cout + n_base + c0);
#pragma unroll
                            for (int k = 0; k < 4; ++k) sc4[k] = __ldg(sp + k);
                        }
                    }
                    float v[16], r[16];
                    tmem_ld16(tmem_base + ((uint32_t)(q * 32) << 16) + buf * Cfg::kAccCols + (mt0 + mt) * N_CTA + c0, v);
                    if (SC) tmem_ld16(tmem_base + ((uint32_t)(q * 32) << 16) + (2 + buf) * Cfg::kAccCols + (mt0 + mt) * N_CTA + c0, r);
                    if (c0 + 16 >= N_CTA && mt == MTH - 1) {
                        // accumulator completely read: hand this TMEM buffer back to the MMA warp
                        tc_fence_before();
                        __syncwarp();
                        if (lane == 0) mbar_arrive(&acc_empty[buf]);
                    }
                    if (!p.bias_mma) {
#pragma unroll
                        for (int i = 0; i < 16; ++i) v[i] += bias_s[n_base + c0 + i];
                    }
                    if (SC && valid) {
                        // the residual as a stand-alone shortcut launch would have stored it (16-bit, fp16 range guard included)
                        const float scv[16] = {sc4[0].x, sc4[0].y, sc4[0].z, sc4[0].w, sc4[1].x, sc4[1].y, sc4[1].z, sc4[1].w,
                                               sc4[2].x, sc4[2].y, sc4[2].z, sc4[2].w, sc4[3].x, sc4[3].y, sc4[3].z, sc4[3].w};
#pragma unroll
                        for (int i = 0; i < 8; ++i) {
                            const uint32_t rw = pack2<BF16>(r[2 * i], r[2 * i + 1]);
                            if (!BF16) track16(rw, omax);
                            const float2 r2 = unpack2<BF16>(rw);
                            v[2 * i] = fmaf(v[2 * i], scv[2 * i], r2.x);
                            v[2 * i + 1] = fmaf(v[2 * i + 1], scv[2 * i + 1], r2.y);
                        }
                    } else if (kLoadRes && valid) {
                        const uint32_t rw[8] = {rv_c[mt][cc].x, rv_c[mt][cc].y, rv_c[mt][cc].z, rv_c[mt][cc].w,
                                                rv_c[mt][cc + 1].x, rv_c[mt][cc + 1].y, rv_c[mt][cc + 1].z, rv_c[mt][cc + 1].w};
                        const float scv[16] = {sc4[0].x, sc4[0].y, sc4[0].z, sc4[0].w, sc4[1].x, sc4[1].y, sc4[1].z, sc4[1].w,
                                               sc4[2].x, sc4[2].y, sc4[2].z, sc4[2].w, sc4[3].x, sc4[3].y, sc4[3].z, sc4[3].w};
#pragma unroll
                        for (int i = 0; i < 8; ++i) {
                            const float2 r2 = unpack2<BF16>(rw[i]);
                            v[2 * i] = fmaf(v[2 * i], scv[2 * i], r2.x);
                            v[2 * i + 1] = fmaf(v[2 * i + 1], scv[2 * i + 1], r2.y);
                        }
                    }
#pragma unroll
                    for (int i = 0; i < 16; ++i) v[i] = fmaxf(v[i], v[i] * slope);
                    auto pack_out = [&](int j) {
                        uint4 o;
                        o.x = valid ? pack2<BF16>(v[j * 8 + 0], v[j * 8 + 1]) : 0u;
                        o.y = valid ? pack2<BF16>(v[j * 8 + 2], v[j * 8 + 3]) : 0u;
                        o.z = valid ? pack2<BF16>(v[j * 8 + 4], v[j * 8 + 5]) : 0u;
                        o.w = valid ? pack2<BF16>(v[j * 8 + 6], v[j * 8 + 7]) : 0u;
                        return o;
                    };
                    if (opix_c[mt] >= 0) {
                        uint16_t* dst = p.out + (size_t)opix_c[mt] * 8 + (size_t)((n_base + c0) >> 3) * plane8;
#pragma unroll
                        for (int j = 0; j < 2; ++j) {
                            const uint4 o = pack_out(j);
                            *reinterpret_cast<uint4*>(dst + j * plane8) = o;
                            if (!BF16) track16(o, omax);
                            if constexpr (kCanSum) {
                                if (do_sums && valid) {
                                    // exactly plane_sum_kernel's arithmetic on the value just stored
                                    const uint32_t ow[4] = {o.x, o.y, o.z, o.w};
#pragma unroll
                                    for (int e = 0; e < 4; ++e) {
                                        float2 f = unpack2<BF16>(ow[e]);
                                        if (BF16) { f.x = fminf(fmaxf(f.x, -65504.f), 65504.f); f.y = fminf(fmaxf(f.y, -65504.f), 65504.f); }
                                        sacc[(c0 + j * 8 + 2 * e) % kSumRegs] += (long long)__float2int_rn(f.x * 32768.f);
                                        sacc[(c0 + j * 8 + 2 * e + 1) % kSumRegs] += (long long)__float2int_rn(f.y * 32768.f);
                                    }
                                }
                            }
                        }
                    }
                    if constexpr (kTSum) {
                        // without pix_sub every valid row is a stored row; the others put zeros in the tile
                        uint4* tile = tot_tile + ((cc / 2) % Cfg::kTotalsTiles) * (Cfg::kTotalsTileBytes / 16);
                        tot.put(tile, lane, 0, pack_out(0));
                        tot.put(tile, lane, 1, pack_out(1));
                        tot.add_chunk(tile, 0, cc / 2, p.sums, p.cout, lane);
                    }
                }
            }
#pragma unroll
            for (int mt = 0; mt < MTH; ++mt) {
                bidx_c[mt] = bidx_n[mt]; opix_c[mt] = opix_n[mt];
                bidx_n[mt] = bidx_nn[mt]; opix_n[mt] = opix_nn[mt];
                if (kLoadRes) {
#pragma unroll
                    for (int k = 0; k < NCH; ++k) rv_c[mt][k] = rv_n[mt][k];
                }
            }
        }
        if (kCanSum && do_sums) flush_sums();
        if constexpr (kTSum) tot.flush(p.sums, p.cout, lane);
        if (!BF16 && p.overflow != nullptr && saturated16(omax)) atomicAdd(p.overflow, 1u);
        } else {
        // ---------------------------------------------------------------- epilogue warps (4..11)
        // two warps per TMEM lane quadrant; each takes half of the item's MT accumulator tiles
        constexpr int MTH = MT / 2;
        const int q = warp & 3;                 // TMEM lane quadrant this warp may read
        const int mt0 = ((warp - 4) >> 2) * MTH;
        uint32_t n_done = 0;
        uint32_t omax = 0u;                     // fp16 range guard: max |x| of what this thread stored
        constexpr int NCH = N_CTA / 8;          // 8-channel chunks per pixel in this N slice
        constexpr int RCH = NCH > 8 ? 8 : NCH;  // chunks per residual prefetch group
        constexpr int NG = NCH / RCH;           // prefetch groups
        // channel totals (transposed ownership, ConvTotals): up to two N splits (cout <= 256), acc[ns * NG + g][cc / 2]
        constexpr bool kTSum = TOT;
        static_assert(!kTSum || MTH == 1, "ConvTotals takes one 32-row block per warp and item");
        static_assert(Cfg::kTotalsTiles == 1, "one tile per warp on the 128-column epilogue");
        ConvTotals<BF16, 2 * NG, RCH / 2, 1> tot;
        uint4* tot_tile = reinterpret_cast<uint4*>(totals_smem + (warp - 4) * Cfg::kTotalsTileBytes);
        if constexpr (kTSum) tot.init();
        int tile_next = item_begin / n_split, ns_next = item_begin % n_split;
        for (int item = item_begin; item < item_end; ++item, ++n_done) {
            const int tile = tile_next, ns = ns_next;
            if (++ns_next == n_split) { ns_next = 0; ++tile_next; }
            const int buf = (int)(n_done & 1);
            const int p0 = p.G + tile * Cfg::kTileM;
            const int n_base = ns * N_CTA;
            // per-pixel bookkeeping for the pixels this thread owns: one coalesced table read each
            int bidx[MTH];
            uint16_t* optr[MTH];
            size_t roff[MTH];                       // residual offset: same pixel as the conv input
#pragma unroll
            for (int mt = 0; mt < MTH; ++mt) {
                const int pix = p0 + (mt0 + mt) * 128 + q * 32 + lane;
                const bool in_range = pix < p.p_end;
                bidx[mt] = in_range ? __ldg(p.pix_b + (pix - p.G)) : -1;
                long long opix = in_range ? (long long)pix : -1;
                if (p.pix_sub != nullptr) opix = in_range ? (long long)__ldg(p.pix_sub + (pix - p.G)) : -1;
                optr[mt] = opix >= 0 ? p.out + (size_t)opix * 8 : nullptr;
                roff[mt] = (size_t)pix * 8;
            }
            const size_t plane8 = (size_t)p.out_plane * 8;
            const size_t rplane8 = (size_t)p.res_plane * 8;
            const float slope = p.act_slope;
            constexpr bool fused = FUSED;
            // Fused SE tail: the residual comes from HBM/L2 (~1 us away).  Fetch it in groups of RCH channel chunks per
            // pixel, the first group BEFORE waiting for the accumulator so its latency hides behind the MMAs.
            uint4 rv[MTH][RCH];
            auto fetch_res = [&](int g) {
#pragma unroll
                for (int mt = 0; mt < MTH; ++mt)
#pragma unroll
                    for (int k = 0; k < RCH; ++k) {
                        rv[mt][k] = make_uint4(0u, 0u, 0u, 0u);
                        if (fused && bidx[mt] >= 0)
                            rv[mt][k] = *reinterpret_cast<const uint4*>(p.res + roff[mt] +
                                                                        (size_t)((n_base >> 3) + g * RCH + k) * rplane8);
                    }
            };
            fetch_res(0);
            if constexpr (kTSum) tot.begin_block(bidx[0], p.sums, p.cout, lane);   // a flush overlaps the MMAs
            mbar_wait(&acc_full[buf], (n_done >> 1) & 1);
            tc_fence_after();
#pragma unroll 1
            for (int g = 0; g < NG; ++g) {
                if (g > 0) fetch_res(g);
#pragma unroll
                for (int cc = 0; cc < RCH; cc += 2) {
                    const int c0 = (g * RCH + cc) * 8;
#pragma unroll
                    for (int mt = 0; mt < MTH; ++mt) {
                        const bool valid = bidx[mt] >= 0;
                        float4 sc4[4];
                        if (fused && valid) {
                            const float4* sp = reinterpret_cast<const float4*>(p.se_scale + (size_t)bidx[mt] * p.cout + n_base + c0);
#pragma unroll
                            for (int k = 0; k < 4; ++k) sc4[k] = __ldg(sp + k);
                        }
                        float v[16];
                        tmem_ld16(tmem_base + ((uint32_t)(q * 32) << 16) + buf * Cfg::kAccCols + (mt0 + mt) * N_CTA + c0, v);
                        if (c0 + 16 >= N_CTA && mt == MTH - 1) {
                            // accumulator completely read: hand this TMEM buffer back to the MMA warp
                            tc_fence_before();
                            __syncwarp();
                            if (lane == 0) mbar_arrive(&acc_empty[buf]);
                        }
                        if (!p.bias_mma) {
#pragma unroll
                            for (int i = 0; i < 16; ++i) v[i] += bias_s[n_base + c0 + i];
                        }
                        if (fused && valid) {
                            const uint32_t rw[8] = {rv[mt][cc].x, rv[mt][cc].y, rv[mt][cc].z, rv[mt][cc].w,
                                                    rv[mt][cc + 1].x, rv[mt][cc + 1].y, rv[mt][cc + 1].z, rv[mt][cc + 1].w};
                            const float scv[16] = {sc4[0].x, sc4[0].y, sc4[0].z, sc4[0].w, sc4[1].x, sc4[1].y, sc4[1].z, sc4[1].w,
                                                   sc4[2].x, sc4[2].y, sc4[2].z, sc4[2].w, sc4[3].x, sc4[3].y, sc4[3].z, sc4[3].w};
#pragma unroll
                            for (int i = 0; i < 8; ++i) {
                                const float2 r2 = unpack2<BF16>(rw[i]);
                                v[2 * i] = fmaf(v[2 * i], scv[2 * i], r2.x);
                                v[2 * i + 1] = fmaf(v[2 * i + 1], scv[2 * i + 1], r2.y);
                            }
                        }
#pragma unroll
                        for (int i = 0; i < 16; ++i) v[i] = fmaxf(v[i], v[i] * slope);
                        auto pack_out = [&](int j) {
                            uint4 o;
                            o.x = valid ? pack2<BF16>(v[j * 8 + 0], v[j * 8 + 1]) : 0u;
                            o.y = valid ? pack2<BF16>(v[j * 8 + 2], v[j * 8 + 3]) : 0u;
                            o.z = valid ? pack2<BF16>(v[j * 8 + 4], v[j * 8 + 5]) : 0u;
                            o.w = valid ? pack2<BF16>(v[j * 8 + 6], v[j * 8 + 7]) : 0u;
                            return o;
                        };
                        if (optr[mt] != nullptr) {
                            uint16_t* dst = optr[mt] + (size_t)((n_base + c0) >> 3) * plane8;
#pragma unroll
                            for (int j = 0; j < 2; ++j) {
                                const uint4 o = pack_out(j);
                                *reinterpret_cast<uint4*>(dst + j * plane8) = o;
                                if (!BF16) track16(o, omax);
                            }
                        }
                        if constexpr (kTSum) {
                            // without pix_sub every valid row is a stored row; the others put zeros in the tile
                            tot.put(tot_tile, lane, 0, pack_out(0));
                            tot.put(tot_tile, lane, 1, pack_out(1));
                            tot.add_chunk(tot_tile, ns * NG + g, cc / 2, p.sums, p.cout, lane);
                        }
                    }
                }
            }
        }
        if constexpr (kTSum) tot.flush(p.sums, p.cout, lane);
        if (!BF16 && p.overflow != nullptr && saturated16(omax)) atomicAdd(p.overflow, 1u);
        }
        tc_fence_before();
    }
    __syncthreads();
    if (warp == 2) {
        tc_fence_after();
        tmem_dealloc<Cfg::kTmemCols>(tmem_base);
    }
}

}  // namespace skb
