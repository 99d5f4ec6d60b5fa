// Trial scoring on tcgen05: S = acc * (ra_i + ca_j + a0) + (r_i + q_j + c0),  acc = E . T^T.
//
// Covers cosine scoring (sidekit/iv_scoring.py:108-109), simplified PLDA (:451-462: model_part +
// seg_part + cst + E Psi T^T, Psi folded into E on the host side), two-covariance scoring
// (:192-205, expanded to the same form) and as-norm (sidekit/score_normalization.py:127-138).
//
// Operands are converted once to fp16 "chunk planes" [D/8][rows][8] (the no-swizzle K-major UMMA
// layout, see conv_umma.cuh) after scaling each matrix by a power of two so its largest entry sits
// near 2^9.  Single-pass mode multiplies the fp16 values; split mode also keeps lo = x - hi and
// issues hi*hi + hi*lo + lo*hi into the same fp32 TMEM accumulator, which restores fp32-class
// accuracy (error ~ 2^-22 relative per product) at 3x the tensor work.  The mode is chosen ON THE
// DEVICE from the operands' row norms (no host sync).
//
// Kernel: persistent CTAs, each owning a contiguous run of (row panel, column tile) pairs in
// panel-major order.  For K <= 256 the 128-row E panel stays resident in tensor memory and 128-column
// T tiles stream through a ring of 64- or 128-wide K stages (1-D bulk copies); for larger K (the dense
// layers of the extractor) E and T chunks stream through the ring together.  Accumulators are
// double-buffered in TMEM so the epilogue of tile i overlaps the MMAs of tile i+1.  The score matrix
// is HBM-write-bound (128 FLOP per output byte at D = 256), so the epilogue transposes each 32x32 block through a
// warp-private shared buffer and every store instruction writes one full 128-byte row segment.
#include "sidekit_b200.h"
#include "common.cuh"
#include "layers.cuh"

#include <cmath>
#include <cstdlib>
#include <vector>

namespace skb {

// ----------------------------------------------------------------------------- operand preparation
// stats[0] = max |x| (as float bits), stats[1] = max row sum of squares (float bits).  blockIdx.y selects the operand, so
// both matrices of a scoring call are scanned by one launch.
// No zeroing and no atomics on the results: every CTA leaves its pair of maxima in a scratch list, the CTA that arrives last
// (a self-resetting ticket) reduces the list and stores stats[] (round 1: memset + 2 atomicMax per CTA; the memset alone was
// 2 us of a 60 us row-panel step).
struct AbsmaxArgs { const float* X[2]; int rows[2]; unsigned* stats[2]; float2* partial[2]; unsigned* ticket[2]; };
constexpr int kAbsmaxWarps = 16;
constexpr int kAbsmaxMaxCtas = 8 * kNumSMs;
__global__ void __launch_bounds__(kAbsmaxWarps * 32) absmax_kernel(const AbsmaxArgs a, int D) {
    // one warp per row (every lane sums its columns lane, lane + 32, ... in order, then a shuffle tree: the row sums do not
    // depend on the launch shape), eight loads in flight per lane
    __shared__ float smx[kAbsmaxWarps], sss[kAbsmaxWarps];
    __shared__ bool s_last;
    pdl_wait();                                        // launched with PDL (common.cuh): the scratch list may still be read
    const float* __restrict__ X = a.X[blockIdx.y];
    const int rows = a.rows[blockIdx.y];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    float mx = 0.f, ssm = 0.f;
    for (int row = blockIdx.x * kAbsmaxWarps + warp; row < rows; row += gridDim.x * kAbsmaxWarps) {
        const float* __restrict__ xr = X + (size_t)row * D;
        float ss = 0.f;
        int k = lane;
        for (; k + 7 * 32 < D; k += 8 * 32) {
            float v[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) v[i] = __ldg(xr + k + 32 * i);
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                mx = fmaxf(mx, fabsf(v[i]));
                ss = fmaf(v[i], v[i], ss);
            }
        }
        for (; k < D; k += 32) {
            const float v = __ldg(xr + k);
            mx = fmaxf(mx, fabsf(v));
            ss = fmaf(v, v, ss);
        }
        ssm = fmaxf(ssm, warp_sum(ss));
    }
    mx = warp_max(mx);
    if (lane == 0) { smx[warp] = mx; sss[warp] = ssm; }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int i = 1; i < kAbsmaxWarps; ++i) { mx = fmaxf(mx, smx[i]); ssm = fmaxf(ssm, sss[i]); }
        a.partial[blockIdx.y][blockIdx.x] = make_float2(mx, ssm);
        __threadfence();
        s_last = atomicAdd(a.ticket[blockIdx.y], 1u) == gridDim.x - 1;
    }
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    mx = 0.f; ssm = 0.f;
    for (int i = threadIdx.x; i < (int)gridDim.x; i += blockDim.x) {
        const float2 v = __ldcg(a.partial[blockIdx.y] + i);
        mx = fmaxf(mx, v.x);
        ssm = fmaxf(ssm, v.y);
    }
    mx = warp_max(mx);
    ssm = warp_max(ssm);
    __syncthreads();                                   // smx / sss were read by thread 0 above
    if (lane == 0) { smx[warp] = mx; sss[warp] = ssm; }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int i = 1; i < kAbsmaxWarps; ++i) { mx = fmaxf(mx, smx[i]); ssm = fmaxf(ssm, sss[i]); }
        a.stats[blockIdx.y][0] = __float_as_uint(mx);
        a.stats[blockIdx.y][1] = __float_as_uint(ssm);
        *a.ticket[blockIdx.y] = 0u;                    // ready for the next launch
    }
}

// e such that max|x| * 2^e lies in [2^9, 2^10) (0 for an all-zero operand)
__device__ __forceinline__ int scale_exponent(const unsigned* stats) {
    const float m = __uint_as_float(stats[0]);
    int e = 0;
    if (m > 0.f) { int fe; frexpf(m, &fe); e = 10 - fe; }
    return e;
}

// 1 or 3 passes.  Single-pass error estimate: fp16 rounding 2^-11 per operand, random-sign accumulation over D terms, and a
// factor 7 for the tail of the largest matrices: on 20 000 x 20 000 unit-norm Gaussian rows the worst entry is the diagonal of
// E = T (a squared norm, whose two roundings per term coincide), about 6 x 2^-11 / sqrt(D); with the factor, unit rows of D < 187
// take three passes and D = 256 / 512 one.  The estimate holds for operands whose fp16 rounding errors are uncorrelated: rows
// whose errors add coherently (one repeated value) can exceed it with one pass, and passes = 3 is the bound for them.
__device__ __forceinline__ int decide_passes(const unsigned* statsE, const unsigned* statsT, int D, float abs_alpha, int passes_req) {
    if (passes_req != 0) return passes_req;
    const float nE = sqrtf(__uint_as_float(statsE[1])), nT = sqrtf(__uint_as_float(statsT[1]));
    const float est = abs_alpha * 4.8828125e-4f * nE * nT * 7.f * rsqrtf((float)D);
    return est < 2.5e-4f ? 1 : 3;
}

// X (rows, D) fp32 -> hi / lo fp16 in 128-row tiles of chunk planes: [rows_pad/128][Dp/8][128][8], so that a whole
// (tile, K range) operand image is one contiguous block = one bulk copy; rows >= `rows` and columns >= D are zero.
// blockIdx.y selects the operand.  The scale exponent is derived from the operand's statistics by every thread (and
// stored once for the GEMM epilogue).
struct PackArgs { const float* X[2]; int rows[2], rows_pad[2]; const unsigned* stats[2]; int* exp_out[2]; uint16_t* hi[2]; uint16_t* lo[2]; };
// One CTA per (128-row tile, 64-column group): the rows are READ along K (8 lanes x 32 bytes per row segment: whole sectors),
// split, transposed through shared memory ([chunk][row] with a row stride of 129 16-byte units: conflict-free both ways) and
// WRITTEN as the tile's eight 2 KB chunk planes.  (Round 1 read with one lane per row -- 1 KB apart -- which cost 26 us for a
// 20 000 x 256 operand, profiles/r02l_score_modes_launches.csv.)
constexpr int kPackRowStride = 129;
__global__ void __launch_bounds__(256) pack_split_kernel(const PackArgs a, int D, int Dp) {
    __shared__ uint4 s_hi[8 * kPackRowStride], s_lo[8 * kPackRowStride];
    pdl_wait();
    const int op = blockIdx.z;
    const int rows = a.rows[op], rows_pad = a.rows_pad[op];
    const int tile = blockIdx.x, jg0 = blockIdx.y * 8;
    const float* __restrict__ X = a.X[op];
    const int e_scale = scale_exponent(a.stats[op]);
    if (tile == 0 && blockIdx.y == 0 && threadIdx.x == 0) a.exp_out[op][0] = e_scale;
    if (tile * 128 >= rows_pad) return;                  // the grid is sized for the larger of the two operands
    const float sc = ldexpf(1.f, e_scale);
    const int jl = threadIdx.x & 7, r0 = threadIdx.x >> 3;
    const int k0 = (jg0 + jl) * 8;
    const bool vec = (D & 3) == 0 && (reinterpret_cast<uintptr_t>(X) & 15) == 0 && k0 + 8 <= D;
    float v[4][8];
#pragma unroll
    for (int ps = 0; ps < 4; ++ps) {
        const int row = tile * 128 + ps * 32 + r0;
#pragma unroll
        for (int e = 0; e < 8; ++e) v[ps][e] = 0.f;
        if (row < rows) {
            const float* src = X + (size_t)row * D + k0;
            if (vec) {
                const float4 x0 = __ldg(reinterpret_cast<const float4*>(src)), x1 = __ldg(reinterpret_cast<const float4*>(src) + 1);
                v[ps][0] = x0.x; v[ps][1] = x0.y; v[ps][2] = x0.z; v[ps][3] = x0.w;
                v[ps][4] = x1.x; v[ps][5] = x1.y; v[ps][6] = x1.z; v[ps][7] = x1.w;
            } else {
#pragma unroll
                for (int e = 0; e < 8; ++e)
                    if (k0 + e < D) v[ps][e] = __ldg(src + e);
            }
        }
    }
#pragma unroll
    for (int ps = 0; ps < 4; ++ps) {
        float h[8], l[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) {
            const float x = v[ps][e] * sc;
            const float hv = __half2float(__float2half_rn(x));
            h[e] = hv;
            l[e] = x - hv;
        }
        uint4 oh, ol;
        oh.x = pack2<false>(h[0], h[1]); oh.y = pack2<false>(h[2], h[3]); oh.z = pack2<false>(h[4], h[5]); oh.w = pack2<false>(h[6], h[7]);
        ol.x = pack2<false>(l[0], l[1]); ol.y = pack2<false>(l[2], l[3]); ol.z = pack2<false>(l[4], l[5]); ol.w = pack2<false>(l[6], l[7]);
        s_hi[jl * kPackRowStride + ps * 32 + r0] = oh;
        s_lo[jl * kPackRowStride + ps * 32 + r0] = ol;
    }
    __syncthreads();
    const int chunks = Dp >> 3;
#pragma unroll
    for (int u = threadIdx.x; u < 8 * 128; u += 256) {
        const int j = u >> 7, row = u & 127;
        const size_t o = (((size_t)tile * chunks + jg0 + j) * 128 + row) * 8;
        *reinterpret_cast<uint4*>(a.hi[op] + o) = s_hi[j * kPackRowStride + row];
        *reinterpret_cast<uint4*>(a.lo[op] + o) = s_lo[j * kPackRowStride + row];
    }
}

// ----------------------------------------------------------------------------- the GEMM
struct ScoreParams {
    const uint16_t *Ehi, *Elo, *Thi, *Tlo;   // [rows_pad/128][Dp/8][128][8]
    int Ne, Nt, Ne_pad, Dp, D;
    const int *expE, *expT;                   // per-operand scale exponents (on the device)
    const unsigned *statsE, *statsT;          // operand statistics: the pass count is decided from them on the device
    float abs_alpha;
    int passes_req;                           // 0 = decide on the device, 1 or 3 = forced
    const float *ra, *ca;                     // multiplicative row / column terms (may be null)
    const float *r, *q;                       // additive row / column terms (may be null)
    float a0, c0, rq_scale;                   // acc * (ra_i + ca_j + a0) * 2^-(eE+eT) + rq_scale * (r_i + q_j) + c0
    int mul_scaled;                           // 1: ra / ca are also divided by the operand scales
    void* out;
    long long ld_out;
    int out_mode;                             // 0 = float32 matrix, 1 = float64 matrix, 2 = float16 matrix, 3 = trial list
    // trial-list mode: only the trials of a mask are written, compacted in row-major order (what the reference selects with
    // scoremat[trialmask], sidekit/nnet/xvector.py:243-245): bit j of mask_words[row][w] = trial (row, 32 w + j),
    // word_off[row][w] = number of trials before (row, 32 w).  out = float32 [n_trials].
    const uint32_t* mask_words;
    const uint32_t* word_off;
    int mask_ld;
    int n_ntiles;
    // top-k mode (out_mode 4): every epilogue warp keeps the best topk_k (score, column) keys of each of its rows among the
    // columns it visits and leaves them, when it moves off a row panel, in out = uint64 [Ne][topk_segs][topk_k] (see
    // topk_segment); topk_merge_kernel selects the final k from those partial lists.
    int topk_k, topk_segs;
};

struct TrialTables { const uint32_t* words; const uint32_t* offsets; int ld, Ne, Nt; };
struct TopkLists { unsigned long long* keys; int k, segs; };

// Epilogue modes of score_gemm_body: the (Ne, Nt) matrix (float32 / float64 / float16), the trials of a mask, or the k best
// columns of every row.
constexpr int kEpiMatrix = 0, kEpiTrials = 1, kEpiTopk = 2;

// The CTA whose contiguous run of work items (score_gemm_body) contains item t, for `tiles` items over `grid` CTAs: the
// largest b with floor(tiles * b / grid) <= t.
__host__ __device__ __forceinline__ int score_cta_of(long long t, int tiles, int grid) {
    return (int)(((t + 1) * grid + tiles - 1) / tiles) - 1;
}
// Top-k mode: the row panel's columns are split over the CTAs whose runs touch the panel and, inside a CTA, over the two
// epilogue warps of a TMEM lane quadrant (64 columns of every tile each).  Partial list slot of (CTA, part) and the number of
// slots of a panel -- both pure functions of the partition, so no atomics and a deterministic result.
__host__ __device__ __forceinline__ int topk_first_cta(int panel, int n_ntiles, int tiles, int grid) {
    return score_cta_of((long long)panel * n_ntiles, tiles, grid);
}
__host__ __device__ __forceinline__ int topk_panel_segs(int panel, int n_ntiles, int tiles, int grid) {
    return 2 * (score_cta_of((long long)(panel + 1) * n_ntiles - 1, tiles, grid) - topk_first_cta(panel, n_ntiles, tiles, grid) + 1);
}

// 64-bit total order of the top-k selection: higher score first, lower column first among equal scores.  f2key maps finite
// floats (and the infinities) order-preservingly onto non-zero 32-bit keys, so key 0 pads a list of fewer than k entries.
__device__ __forceinline__ unsigned f2key(float f) {   // order-preserving float -> uint
    const unsigned u = __float_as_uint(f);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float key2f(unsigned k) {
    const unsigned u = (k & 0x80000000u) ? (k & 0x7fffffffu) : ~k;
    return __uint_as_float(u);
}
__device__ __forceinline__ unsigned long long topk_key(float s, int col) {
    return ((unsigned long long)f2key(s) << 32) | (unsigned)~col;
}
// One lane's k best keys as a binary min-heap in a warp's [k][32] shared-memory lists (slot s of lane l at h[32 s + l]: the
// lanes of a warp touch the same 256 bytes whatever slots they are at).  Replaces the root (the current k-th best) with a
// larger key and restores the heap; returns the new root.  log2(k) levels instead of a rescan of all k slots.
__device__ __forceinline__ unsigned long long topk_heap_replace(unsigned long long* h, int lane, int k, unsigned long long key) {
    int i = 0;
    for (;;) {
        int c = 2 * i + 1;
        if (c >= k) break;
        unsigned long long kc = h[c * 32 + lane];
        if (c + 1 < k) {
            const unsigned long long kr = h[(c + 1) * 32 + lane];
            if (kr < kc) { kc = kr; ++c; }
        }
        if (key <= kc) break;
        h[i * 32 + lane] = kc;
        i = c;
    }
    h[i * 32 + lane] = key;
    return h[lane];
}
// the float threshold a score has to reach before its key is built and compared (-inf while the list has free slots)
__device__ __forceinline__ float topk_screen(unsigned long long kth) {
    const unsigned hi = (unsigned)(kth >> 32);
    return hi ? key2f(hi) : -INFINITY;
}

constexpr int kScKChunk = 64;

// smem: [ctrl 256 B][E staging piece][B ring][8 warps x [32][36] fp32 transpose buffers]
// KC = K elements per ring stage of the single-pass resident-panel variant (64 or 128).  Every tcgen05.commit costs the
// tensor pipe a drain of ~140 ns (the MMAs behind it do not start before the ones in front have completed): with 64-wide
// stages a 128 x 128 x 256 tile is 4 x (4 MMAs + commit) and the pipe idles 60 % of the time; 128-wide stages (8 MMAs per
// commit, 32 KB bulk copies) take the MMA-only time of a 20k x 20k call from 0.246 to 0.200 ms
// (profiles/r02x_score_issue_bound.txt).
constexpr int kKc128Stages = 3;   // 32 KB stages of the 128-wide variant (4 fit since the E panel is staged through 32 KB, and are slower: profiles/r02x_score_issue_bound.txt)
constexpr int kAPieceK = 128;     // E staging piece: 128 K-columns (32 KB) measured faster than 64 and 32 (profiles/r02x_score_issue_bound.txt)
template <int PASSES, bool STREAM_A, int KC = 64>
struct ScoreSmem {
    static constexpr int kParts = PASSES == 1 ? 1 : 2;
    static_assert(KC == 64 || (KC == 128 && PASSES == 1 && !STREAM_A), "128-wide stages: single-pass resident-panel variant only");
    static constexpr int kChunk = PASSES == 1 ? KC : 32;              // K elements per stage
    static constexpr int kStageBytes = 128 * kChunk * 2;              // one part (hi or lo) of one operand of one stage
    // resident-panel mode: a stage holds a T chunk; streaming mode (large K): an E chunk and a T chunk
    static constexpr int kRingStageBytes = (STREAM_A ? 2 : 1) * kParts * kStageBytes;
    static constexpr int kEpiWarps = 8;
    static constexpr int kThreads = (2 + kEpiWarps) * 32;  // warps: 0 producer, 1 MMA, 2.. epilogue (two per TMEM quadrant)
    static constexpr int kBStages = STREAM_A ? 4 : (PASSES == 3 ? 3 : (KC == 128 ? kKc128Stages : 7));
    // Resident-panel variants keep the E panel in TENSOR memory (copied there once per panel with tcgen05.cp): a tcgen05.mma
    // then reads only the T tile through the shared-memory pipe.  With both operands in shared memory a 128 x 128 x 256 tile
    // moved 128 KB of operand reads + 64 KB of incoming T + 64-128 KB of epilogue staging through a 128 B/clk pipe: 2000-2500
    // cycles against 1024 of math -- every output mode was bound by shared-memory bandwidth (profiles/r02x_score_smem_bound.txt).
    static constexpr bool kATmem = !STREAM_A;
    static constexpr int kAccCols = 2 * 128;             // double-buffered accumulators
    static constexpr int kTmemCols = kATmem ? 512 : kAccCols;   // + kParts x 128 columns of A (Dp <= 256)
    static constexpr int kStageRowBytes = 36 * 4;        // [32][36] fp32 transpose buffer per epilogue warp (16-byte rows)
    // the E panel passes into tensor memory piece by piece through a staging piece of kAPieceK K-columns of one part
    static constexpr size_t kABytes = kATmem ? (size_t)128 * kAPieceK * 2 : 0;
    // Epilogue region: the warps' [32][36] transpose buffers, or in top-k mode (topk_k > 0, lane = row: no transpose) the
    // warps' [topk_k][32] lists of 64-bit keys in their place -- 64 KB at k = 32, which the KC 64 ring would not fit next to
    // the 36 KB of buffers.
    static size_t epi_bytes(int topk_k) {
        return topk_k > 0 ? (size_t)kEpiWarps * 32 * topk_k * sizeof(unsigned long long) : (size_t)kEpiWarps * 32 * kStageRowBytes;
    }
    static size_t total(int topk_k) { return 256 + kABytes + (size_t)kBStages * kRingStageBytes + epi_bytes(topk_k); }
};

#ifdef SKB_SCORE_TIMING
// diagnostic build only (./build.sh -DSKB_SCORE_TIMING): where do the roles of score_gemm_kernel wait?  Cycles summed over CTAs.
__device__ unsigned long long g_score_t[16];
#define SKB_T0() const long long t0__ = clock64()
#define SKB_TADD(i) atomicAdd(&g_score_t[i], (unsigned long long)(clock64() - t0__))
#define SKB_TIMED_WAIT(i, stmt) do { const long long tw__ = clock64(); stmt; if ((threadIdx.x & 31) == 0) atomicAdd(&g_score_t[i], (unsigned long long)(clock64() - tw__)); } while (0)
#else
#define SKB_T0()
#define SKB_TADD(i)
#define SKB_TIMED_WAIT(i, stmt) stmt
#endif

template <int PASSES, bool STREAM_A, int MODE, int KC = 64>
__device__ __forceinline__ void score_gemm_body(const ScoreParams& p) {
    using SM = ScoreSmem<PASSES, STREAM_A, KC>;
    static_assert(MODE != kEpiTopk || !STREAM_A, "top-k mode: resident-panel variants only");
    constexpr bool TRIALS = MODE == kEpiTrials, TOPK = MODE == kEpiTopk;
    extern __shared__ __align__(128) uint8_t smem[];
    uint64_t* a_full = reinterpret_cast<uint64_t*>(smem);
    uint64_t* a_empty = a_full + 1;
    uint64_t* b_full = a_empty + 1;                 // [kBStages]
    uint64_t* b_empty = b_full + SM::kBStages;      // [kBStages]
    uint64_t* acc_full = b_empty + SM::kBStages;    // [2]
    uint64_t* acc_empty = acc_full + 2;             // [2]
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + 2);
    uint8_t* a_smem = smem + 256;
    uint8_t* b_smem = a_smem + SM::kABytes;
    uint8_t* stage_smem = b_smem + SM::kBStages * SM::kRingStageBytes;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    // contiguous run of work items for this CTA (panel-major), walked with incremental (panel, nt) counters; an item = one
    // 128-row panel x one 128-column tile
    const int n_panels = p.Ne_pad >> 7;
    const int tiles_total = n_panels * p.n_ntiles;
    const int t_begin = (int)((long long)tiles_total * blockIdx.x / gridDim.x);
    const int t_end = (int)((long long)tiles_total * (blockIdx.x + 1) / gridDim.x);
    const int panel0 = t_begin / p.n_ntiles, nt0 = t_begin % p.n_ntiles;
    const int n_kc = p.Dp / SM::kChunk;

    if (threadIdx.x == 0) {
        mbar_init(a_full, 1);
        mbar_init(a_empty, 1);
        for (int i = 0; i < SM::kBStages; ++i) { mbar_init(&b_full[i], 1); mbar_init(&b_empty[i], 1); }
        for (int i = 0; i < 2; ++i) { mbar_init(&acc_full[i], 1); mbar_init(&acc_empty[i], SM::kEpiWarps); }
        fence_barrier_init();
    }
    if (warp == 1) tmem_alloc<SM::kTmemCols>(tmem_slot);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        // ---------------------------------------------------------------- producer: E panel (on change) + T chunks
        if (lane == 0) {
            SKB_T0();
            int panel = panel0, nt = nt0, s = 0;
            uint32_t b_ph = 1, a_ph = 1;
            bool new_panel = true;
            for (int t = t_begin; t < t_end; ++t) {
                if (SM::kATmem && new_panel) {
                    // piece by piece through the staging buffer (the MMA lane copies each piece on into tensor memory)
                    for (int part = 0; part < SM::kParts; ++part)
                        for (int k0 = 0; k0 < p.Dp; k0 += kAPieceK) {
                            mbar_wait(a_empty, a_ph);
                            a_ph ^= 1;
                            const uint32_t bytes = (uint32_t)min(kAPieceK, p.Dp - k0) * 256u;       // 128 rows x 2 bytes per K column
                            mbar_arrive_expect_tx(a_full, bytes);
                            bulk_g2s(a_smem, (part == 0 ? p.Ehi : p.Elo) + (size_t)panel * p.Dp * 128 + (size_t)k0 * 128, bytes, a_full);
                        }
                }
                for (int kc = 0; kc < n_kc; ++kc) {
                    SKB_TIMED_WAIT(4, mbar_wait(&b_empty[s], b_ph));
                    mbar_arrive_expect_tx(&b_full[s], SM::kRingStageBytes);
                    uint8_t* dst = b_smem + (size_t)s * SM::kRingStageBytes;
                    if (STREAM_A) {
                        for (int part = 0; part < SM::kParts; ++part, dst += SM::kStageBytes) {
                            const uint16_t* src = (part == 0 ? p.Ehi : p.Elo) + ((size_t)panel * p.Dp + (size_t)kc * SM::kChunk) * 128;
                            bulk_g2s(dst, src, SM::kStageBytes, &b_full[s]);
                        }
                    }
                    for (int part = 0; part < SM::kParts; ++part, dst += SM::kStageBytes) {
                        const uint16_t* src = (part == 0 ? p.Thi : p.Tlo) + ((size_t)nt * p.Dp + (size_t)kc * SM::kChunk) * 128;
                        bulk_g2s(dst, src, SM::kStageBytes, &b_full[s]);   // contiguous planes
                    }
                    if (++s == SM::kBStages) { s = 0; b_ph ^= 1; }
                }
                new_panel = false;
                if (++nt == p.n_ntiles) { nt = 0; ++panel; new_panel = true; }
            }
            SKB_TADD(7);
        }
    } else if (warp == 1) {
        // ---------------------------------------------------------------- MMA issuer: ONE lane runs the whole loop
        // (The tensor pipe needs 256 cycles for the four MMAs of a stage; with a warp-uniform loop -- every lane polling the
        // barriers, elect.sync + __syncwarp around each stage -- the issue path took ~800 cycles per stage and the pipe idled
        // two thirds of the time: tools/score_timing_probe.py, profiles/r02x_score_issue_bound.txt.)
        if (lane == 0) {
        const uint32_t idesc = umma_idesc_f16(128, 128, false);
        const uint64_t desc_hi = (static_cast<uint64_t>(2048 >> 4) << 16) | (static_cast<uint64_t>(128 >> 4) << 32) |
                                 (static_cast<uint64_t>(1) << 46);
        int nt = nt0, s = 0;
        uint32_t b_ph = 0, a_ph = 0, nt_done = 0;
        bool new_panel = true;
        SKB_T0();
        for (int t = t_begin; t < t_end; ++t, ++nt_done) {
            if (SM::kATmem && new_panel) {
                // the panel moves on into tensor memory piece by piece (behind the MMAs of the previous panel, which execute
                // first: one in-order pipe); the staging buffer is free again as soon as a piece's copies are done
                for (int part = 0; part < SM::kParts; ++part)
                    for (int k0 = 0; k0 < p.Dp; k0 += kAPieceK) {
                        SKB_TIMED_WAIT(3, mbar_wait(a_full, a_ph));
                        a_ph ^= 1;
                        tc_fence_after();
                        const int n_ks = min(kAPieceK, p.Dp - k0) / 16;
                        for (int ks = 0; ks < n_ks; ++ks)
                            tmem_cp_128x256b(tmem_base + SM::kAccCols + part * 128 + (k0 / 16 + ks) * 8,
                                             desc_hi | (((smem_u32(a_smem) + ks * 2 * 2048) >> 4) & 0x3FFF));
                        umma_commit(a_empty);
                    }
            }
            const int buf = (int)(nt_done & 1);
            SKB_TIMED_WAIT(2, mbar_wait(&acc_empty[buf], ((nt_done >> 1) & 1) ^ 1));
            tc_fence_after();
            const uint32_t d_tmem = tmem_base + buf * 128;
            for (int kc = 0; kc < n_kc; ++kc) {
                SKB_TIMED_WAIT(1, mbar_wait(&b_full[s], b_ph));
                tc_fence_after();
                // streaming mode: the stage holds the E chunk (hi, lo) in front of the T chunk
                const uint32_t st_base = smem_u32(b_smem + (size_t)s * SM::kRingStageBytes);
                const uint32_t b_hi = st_base + (STREAM_A ? SM::kParts * SM::kStageBytes : 0);
#pragma unroll
                for (int combo = 0; combo < (PASSES == 1 ? 1 : 3); ++combo) {
                    // combo 0: hi*hi, 1: hi*lo, 2: lo*hi
                    const uint32_t a_b = st_base + (combo == 2 ? SM::kStageBytes : 0);
                    const uint32_t b_b = b_hi + (combo == 1 ? SM::kStageBytes : 0);
#pragma unroll
                    for (int ks = 0; ks < SM::kChunk / 16; ++ks) {
                        const uint64_t bd = desc_hi | (((b_b + ks * 2 * 2048) >> 4) & 0x3FFF);
                        const uint32_t acc = (kc > 0 || combo > 0 || ks > 0) ? 1u : 0u;
                        if (SM::kATmem) {
                            umma_f16_ts(d_tmem, tmem_base + SM::kAccCols + (combo == 2 ? 128 : 0) + (kc * (SM::kChunk / 16) + ks) * 8, bd, idesc, acc);
                        } else {
                            const uint64_t ad = desc_hi | (((a_b + ks * 2 * 2048) >> 4) & 0x3FFF);
                            umma_f16(d_tmem, ad, bd, idesc, acc);
                        }
                    }
                }
                umma_commit(&b_empty[s]);
                if (++s == SM::kBStages) { s = 0; b_ph ^= 1; }
            }
            new_panel = false;
            if (++nt == p.n_ntiles) { nt = 0; new_panel = true; }
            umma_commit(&acc_full[buf]);
        }
        SKB_TADD(0);
        }
        __syncwarp();
    } else if (warp >= 2) {
        // ---------------------------------------------------------------- epilogue: two warps per TMEM lane quadrant
        constexpr int NB = 2;                              // 32-column blocks per warp and tile
        const int q = warp & 3;
        const int part = (warp - 2) >> 2;                  // which NB of the four 32-column blocks
        float* stg = reinterpret_cast<float*>(stage_smem) + (warp - 2) * 32 * 36;   // warp-private [32][36] transpose buffer
        const int esz = p.out_mode == 1 ? 8 : (p.out_mode == 2 ? 2 : 4);
        // top-k mode: this warp's [k][32] lists (over the transpose buffers, which the mode does not use), and per lane the
        // k-th best key of its row so far
        unsigned long long* lst = reinterpret_cast<unsigned long long*>(stage_smem) + (size_t)(warp - 2) * 32 * (TOPK ? p.topk_k : 0);
        unsigned long long kth = 0ull;
        float kth_f = -INFINITY;
        if (TOPK)
            for (int s = 0; s < p.topk_k; ++s) lst[s * 32 + lane] = 0ull;
        const bool out_ok = p.out_mode >= 3 ? true
                          : p.out_mode == 2 ? ((p.ld_out * 2) % 8 == 0 && (reinterpret_cast<uintptr_t>(p.out) & 7) == 0)
                                            : ((p.ld_out * esz) % 16 == 0 && (reinterpret_cast<uintptr_t>(p.out) & 15) == 0);
        const bool vec_ok = out_ok && (p.q == nullptr || (reinterpret_cast<uintptr_t>(p.q) & 15) == 0);
        const float inv_scale = ldexpf(1.f, -(p.expE[0] + p.expT[0]));
        const float a0 = p.a0 * inv_scale;
        const float mscale = p.mul_scaled ? inv_scale : 1.f;
        int panel = panel0, nt = nt0;
        uint32_t nt_done = 0;
        SKB_T0();
        // Row terms change only with the panel; column terms are fetched BEFORE waiting for the accumulator, so their
        // L2 latency hides behind the MMAs instead of stalling every 32x32 block (was 52 % of all stall samples).
        int cur_panel = -1;
        float ra = 0.f, rr = 0.f;
        const int c4 = (lane & 7) * 4;
        uint32_t mwn[NB], mon[NB];                         // trial-list mode: mask words / offsets of the NEXT item
        auto fetch_mask = [&](int pnl, int ntile) {
            const int rown = pnl * 128 + q * 32 + lane;
#pragma unroll
            for (int cbi = 0; cbi < NB; ++cbi) {
                const int wcol = ntile * 4 + part * NB + cbi;
                mwn[cbi] = 0u; mon[cbi] = 0u;
                if (rown < p.Ne && wcol < p.mask_ld) {
                    mwn[cbi] = __ldg(p.mask_words + (size_t)rown * p.mask_ld + wcol);
                    mon[cbi] = __ldg(p.word_off + (size_t)rown * p.mask_ld + wcol);
                }
            }
        };
#pragma unroll
        for (int cbi = 0; cbi < NB; ++cbi) { mwn[cbi] = 0u; mon[cbi] = 0u; }
        if (TRIALS && t_begin < t_end) fetch_mask(panel0, nt0);
        float4 qnext[NB];
        auto fetch_q = [&](int ntile) {
#pragma unroll
            for (int cbi = 0; cbi < NB; ++cbi) {
                const int col = ntile * 128 + (part * NB + cbi) * 32 + c4;
                qnext[cbi] = make_float4(0.f, 0.f, 0.f, 0.f);
                if (p.q && vec_ok && col + 4 <= p.Nt) qnext[cbi] = __ldg(reinterpret_cast<const float4*>(p.q + col));
            }
        };
#pragma unroll
        for (int cbi = 0; cbi < NB; ++cbi) qnext[cbi] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (t_begin < t_end) fetch_q(nt0);
        for (int t = t_begin; t < t_end; ++t, ++nt_done) {
            const int buf = (int)(nt_done & 1);
            if (panel != cur_panel) {
                cur_panel = panel;
                const int r = panel * 128 + q * 32 + lane;
                ra = (p.ra && r < p.Ne) ? p.ra[r] * mscale : 0.f;
                rr = fmaf((p.r && r < p.Ne) ? p.r[r] : 0.f, p.rq_scale, p.c0);
            }
            // column terms: fetched ONE ITEM AHEAD as well (fetched at the top of their own tile they were the first thing the
            // epilogue stalled on whenever the accumulator was already waiting: 15 % of the stall samples)
            float4 qpre[NB];
#pragma unroll
            for (int cbi = 0; cbi < NB; ++cbi) qpre[cbi] = qnext[cbi];
            {
                int ntn = nt + 1;
                if (ntn == p.n_ntiles) ntn = 0;
                if (t + 1 < t_end) fetch_q(ntn);
            }
            // trial-list mode: lane = row (the accumulator's native layout, no transpose): this row's mask words and output
            // offsets, fetched ONE ITEM AHEAD (a mask word comes from L2 / HBM, ~1 us away: loaded at the top of its own tile it
            // was 36 % of the kernel's stall samples and the tensor pipe sat at 4 %)
            uint32_t mw[NB], mo[NB];
#pragma unroll
            for (int cbi = 0; cbi < NB; ++cbi) { mw[cbi] = mwn[cbi]; mo[cbi] = mon[cbi]; }
            if (TRIALS && t + 1 < t_end) {
                int ntn = nt + 1, pn = panel;
                if (ntn == p.n_ntiles) { ntn = 0; ++pn; }
                fetch_mask(pn, ntn);
            }
            if (warp == 2) { SKB_TIMED_WAIT(5, mbar_wait(&acc_full[buf], (nt_done >> 1) & 1)); }
            else mbar_wait(&acc_full[buf], (nt_done >> 1) & 1);
            tc_fence_after();
            const int row0 = panel * 128 + q * 32;
            const int n_rows = min(32, p.Ne - row0);
#pragma unroll
            for (int cbi = 0; cbi < NB; ++cbi) {
                const int cb = part * NB + cbi;
                const int col0 = nt * 128 + cb * 32;
                float v[32];
                tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + buf * 128 + cb * 32, v);
                if (cbi == NB - 1) {   // this warp's share of the accumulators is read: release the TMEM buffer
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&acc_empty[buf]);
                }
                if (col0 >= p.Nt || n_rows <= 0) continue;
                if (TOPK) {
                    // lane = row (the accumulator's native layout): the lane screens the 32 scores of its row against its
                    // k-th best so far; only a score that reaches it builds a key and touches shared memory.  Same roundings
                    // as the matrix path, so a selected value equals its score_matrix entry bit for bit.
                    const float mul = ra + a0;
                    const int jmax = min(32, p.Nt - col0);
                    // the scaled column term of column col0 + lane: from the prefetched float4s (lane l of the first eight
                    // holds columns 4l .. 4l + 3), or loaded here at a ragged edge / for an unaligned column term
                    float ql;
                    if (p.q != nullptr && vec_ok && jmax == 32) {
                        const float4 qv = qpre[cbi];
                        const float x = __shfl_sync(0xffffffffu, qv.x, lane >> 2), y = __shfl_sync(0xffffffffu, qv.y, lane >> 2);
                        const float z = __shfl_sync(0xffffffffu, qv.z, lane >> 2), w = __shfl_sync(0xffffffffu, qv.w, lane >> 2);
                        const int c = lane & 3;
                        ql = __fmul_rn(c == 0 ? x : (c == 1 ? y : (c == 2 ? z : w)), p.rq_scale);
                    } else {
                        ql = __fmul_rn((p.q != nullptr && lane < jmax) ? __ldg(p.q + col0 + lane) : 0.f, p.rq_scale);
                    }
#pragma unroll
                    for (int j = 0; j < 32; ++j) {
                        const float s = __fadd_rn(fmaf(v[j], mul, rr), __shfl_sync(0xffffffffu, ql, j));
                        if (j < jmax && s >= kth_f) {
                            const unsigned long long key = topk_key(s, col0 + j);
                            if (key > kth) {
                                kth = topk_heap_replace(lst, lane, p.topk_k, key);
                                kth_f = topk_screen(kth);
                            }
                        }
                    }
                    continue;
                }
                if (TRIALS) {
                    // Only the trials of the mask are written, compacted in row-major order: each lane walks the set bits
                    // of ITS row's word (lane = row, the accumulator's native layout: no transpose).  A block without any
                    // trial costs a TMEM load and a vote; otherwise the rows are parked in the warp's staging buffer so that
                    // the set bits can index them.  (Almost) no stores for a sparse mask: the kernel is then bound by the
                    // operand stream / the tensor pipe instead of the HBM write.
                    uint32_t word = mw[cbi];
                    if (__any_sync(0xffffffffu, word != 0u)) {
                        __syncwarp();
                        float4* srow = reinterpret_cast<float4*>(stg + lane * 36);
#pragma unroll
                        for (int k = 0; k < 8; ++k) srow[k] = make_float4(v[4 * k], v[4 * k + 1], v[4 * k + 2], v[4 * k + 3]);
                        // the block's 32 (scaled) column terms ride in the 4 pad floats of the first 8 staging rows: they were
                        // fetched before the accumulator wait (qpre); looked up with a dependent __ldg per trial they were 43 %
                        // of the kernel's stall samples (profiles/r02x_ncu_score_triallist.txt)
                        const bool q_staged = p.q != nullptr && vec_ok && col0 + 32 <= p.Nt;
                        if (q_staged && lane < 8) {
                            const float4 qv = qpre[cbi];
                            *reinterpret_cast<float4*>(stg + lane * 36 + 32) =
                                make_float4(__fmul_rn(qv.x, p.rq_scale), __fmul_rn(qv.y, p.rq_scale), __fmul_rn(qv.z, p.rq_scale), __fmul_rn(qv.w, p.rq_scale));
                        }
                        __syncwarp();
                        const float mul = ra + a0;
                        float* o = reinterpret_cast<float*>(p.out) + mo[cbi];
                        while (word != 0u) {
                            const int j = __ffs(word) - 1;
                            word &= word - 1u;
                            // the same roundings as the matrix path (product, then sum: no contraction into an FMA)
                            const float qq = q_staged ? stg[(j >> 2) * 36 + 32 + (j & 3)]
                                                      : (p.q ? __fmul_rn(__ldg(p.q + col0 + j), p.rq_scale) : 0.f);
                            *o++ = __fadd_rn(fmaf(stg[lane * 36 + j], mul, rr), qq);
                        }
                    }
                    continue;
                }
                // Transpose through shared memory: lane = row before the transpose (row terms applied there),
                // lane = 4 columns x 1 of 4 rows after it, so every store instruction writes four 128-byte row segments.
                __syncwarp();
                // rows beyond Ne (the last panel of a ragged matrix) are simply not stored: the ragged panel used to take the
                // scalar path and its CTA finished several times later than all the others
                const bool fast = (p.ca == nullptr) && col0 + 32 <= p.Nt && vec_ok;
                if (fast) {
                    const float mul = ra + a0;
                    float4* srow = reinterpret_cast<float4*>(stg + lane * 36);
#pragma unroll
                    for (int k = 0; k < 8; ++k)
                        srow[k] = make_float4(fmaf(v[4 * k], mul, rr), fmaf(v[4 * k + 1], mul, rr), fmaf(v[4 * k + 2], mul, rr),
                                              fmaf(v[4 * k + 3], mul, rr));
                    __syncwarp();
                    const int rs = lane >> 3;
                    // explicit roundings (product, then sum) so that every output mode performs the same arithmetic
                    float4 qv = qpre[cbi];
                    qv.x = __fmul_rn(qv.x, p.rq_scale); qv.y = __fmul_rn(qv.y, p.rq_scale);
                    qv.z = __fmul_rn(qv.z, p.rq_scale); qv.w = __fmul_rn(qv.w, p.rq_scale);
                    if (p.out_mode == 2) {
                        __half* o = reinterpret_cast<__half*>(p.out) + (size_t)(row0 + rs) * p.ld_out + col0 + c4;
                        const size_t step = (size_t)4 * p.ld_out;
#pragma unroll
                        for (int it = 0; it < 8; ++it, o += step) {
                            if (it * 4 + rs >= n_rows) break;
                            const float4 x = *reinterpret_cast<const float4*>(stg + (it * 4 + rs) * 36 + c4);
                            const __half2 h0 = __floats2half2_rn(__fadd_rn(x.x, qv.x), __fadd_rn(x.y, qv.y)), h1 = __floats2half2_rn(__fadd_rn(x.z, qv.z), __fadd_rn(x.w, qv.w));
                            __stcs(reinterpret_cast<uint2*>(o), make_uint2(*reinterpret_cast<const uint32_t*>(&h0), *reinterpret_cast<const uint32_t*>(&h1)));
                        }
                    } else if (p.out_mode == 1) {
                        double* o = reinterpret_cast<double*>(p.out) + (size_t)(row0 + rs) * p.ld_out + col0 + c4;
                        const size_t step = (size_t)4 * p.ld_out;
#pragma unroll
                        for (int it = 0; it < 8; ++it, o += step) {
                            if (it * 4 + rs >= n_rows) break;
                            const float4 x = *reinterpret_cast<const float4*>(stg + (it * 4 + rs) * 36 + c4);
                            __stcs(reinterpret_cast<double2*>(o), make_double2((double)__fadd_rn(x.x, qv.x), (double)__fadd_rn(x.y, qv.y)));
                            __stcs(reinterpret_cast<double2*>(o) + 1, make_double2((double)__fadd_rn(x.z, qv.z), (double)__fadd_rn(x.w, qv.w)));
                        }
                    } else {
                        float* o = reinterpret_cast<float*>(p.out) + (size_t)(row0 + rs) * p.ld_out + col0 + c4;
                        const size_t step = (size_t)4 * p.ld_out;
#pragma unroll
                        for (int it = 0; it < 8; ++it, o += step) {
                            if (it * 4 + rs >= n_rows) break;
                            const float4 x = *reinterpret_cast<const float4*>(stg + (it * 4 + rs) * 36 + c4);
                            // streaming store: the score matrix is written once and never re-read by this kernel, so it
                            // should not evict the T operand tiles from L2
                            __stcs(reinterpret_cast<float4*>(o), make_float4(__fadd_rn(x.x, qv.x), __fadd_rn(x.y, qv.y), __fadd_rn(x.z, qv.z), __fadd_rn(x.w, qv.w)));
                        }
                    }
                    continue;
                }
                // generic path: ragged tile edges, unaligned outputs, or the as-norm form whose column term also
                // multiplies the accumulator
                if (p.ca == nullptr) {
                    const float mul = ra + a0;
#pragma unroll
                    for (int i = 0; i < 32; ++i) stg[lane * 36 + i] = fmaf(v[i], mul, rr);
                } else {
#pragma unroll
                    for (int i = 0; i < 32; ++i) stg[lane * 36 + i] = v[i];
                }
                __syncwarp();
                const int col = col0 + lane;
                const bool col_ok = col < p.Nt;
                const float qq = __fmul_rn((p.q && col_ok) ? __ldg(p.q + col) : 0.f, p.rq_scale);
                const float ca = (p.ca && col_ok) ? __ldg(p.ca + col) * mscale : 0.f;
                float* o = reinterpret_cast<float*>(p.out) + (size_t)row0 * p.ld_out + col;
                double* od = reinterpret_cast<double*>(p.out) + (size_t)row0 * p.ld_out + col;
                __half* oh = reinterpret_cast<__half*>(p.out) + (size_t)row0 * p.ld_out + col;
#pragma unroll 4
                for (int r = 0; r < 32; ++r) {
                    float sv = stg[r * 36 + lane];
                    if (p.ca != nullptr) {
                        const float ra_r = __shfl_sync(0xffffffffu, ra, r), rr_r = __shfl_sync(0xffffffffu, rr, r);
                        sv = fmaf(sv, ra_r + ca + a0, rr_r);
                    }
                    sv = __fadd_rn(sv, qq);
                    if (r < n_rows && col_ok) {
                        if (p.out_mode == 2) oh[(size_t)r * p.ld_out] = __float2half_rn(sv);
                        else if (p.out_mode == 1) od[(size_t)r * p.ld_out] = (double)sv;
                        else o[(size_t)r * p.ld_out] = sv;
                    }
                }
            }
            if (TOPK && (nt + 1 == p.n_ntiles || t + 1 == t_end)) {
                // leaving the row panel: this warp's lists become the partial lists of its segment, and start over empty
                const int row = panel * 128 + q * 32 + lane;
                const int seg = 2 * ((int)blockIdx.x - topk_first_cta(panel, p.n_ntiles, tiles_total, (int)gridDim.x)) + part;
                unsigned long long* dst = reinterpret_cast<unsigned long long*>(p.out) + ((size_t)row * p.topk_segs + seg) * p.topk_k;
                for (int s = 0; s < p.topk_k; ++s) {
                    if (row < p.Ne) dst[s] = lst[s * 32 + lane];
                    lst[s * 32 + lane] = 0ull;
                }
                kth = 0ull;
                kth_f = -INFINITY;
            }
            if (++nt == p.n_ntiles) { nt = 0; ++panel; }
        }
        if (warp == 2 && lane == 0) { SKB_TADD(6); }
    }
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc<SM::kTmemCols>(tmem_base);
    }
}

// ONE launch per call runs the body of the pass count decide_passes returns: forced, or decided from the operand statistics
// (uniform across the grid).  Round 1 launched both pass variants and let one of them return at once: a 3 us no-op per
// call, 5 % of a 2500-row panel at 8 GPUs.  Three-pass bodies use 32-wide stages whatever KC.
template <bool STREAM_A, int MODE, int KC>
__global__ void __launch_bounds__(ScoreSmem<1, STREAM_A>::kThreads, 1) score_gemm_kernel(const ScoreParams p) {
    pdl_wait();                                        // the operand statistics / planes come from the kernels before this one
    if (decide_passes(p.statsE, p.statsT, p.D, p.abs_alpha, p.passes_req) == 1) score_gemm_body<1, STREAM_A, MODE, KC>(p);
    else score_gemm_body<3, STREAM_A, MODE>(p);
}

// ----------------------------------------------------------------------------- packed operands, workspace, launch
struct ScoreWorkspace {
    uint16_t* planes = nullptr;
    size_t planes_cap = 0;
    unsigned* stats = nullptr;   // 2 x (2 stats + 1 exponent) + passes
    float2* partial = nullptr;   // absmax_kernel: per-CTA maxima of the two operands of a call
    unsigned* ticket = nullptr;  // absmax_kernel: arrival counters (zero between launches)
    float* tmp = nullptr;        // scratch score matrix (as-norm cohort scores)
    size_t tmp_cap = 0;
};
// one workspace per (host thread, device): the buffers are cudaMalloc'd on the device that is current at first use
static thread_local ScoreWorkspace g_ws_dev[kMaxDevices];
#define g_ws (g_ws_dev[current_device()])

static int ws_ensure(size_t plane_bytes, size_t tmp_bytes) {
    if (!g_ws.stats) SKB_CUDA_CHECK(cudaMalloc(&g_ws.stats, 8 * sizeof(unsigned)));
    if (!g_ws.partial) SKB_CUDA_CHECK(cudaMalloc(&g_ws.partial, 2 * (size_t)kAbsmaxMaxCtas * sizeof(float2)));
    if (!g_ws.ticket) {
        SKB_CUDA_CHECK(cudaMalloc(&g_ws.ticket, 2 * sizeof(unsigned)));
        SKB_CUDA_CHECK(cudaMemset(g_ws.ticket, 0, 2 * sizeof(unsigned)));
    }
    if (plane_bytes > g_ws.planes_cap) {
        if (getenv("SKB_TRACE_ALLOC")) fprintf(stderr, "skb: scoring plane workspace grows %zu -> %zu bytes\n", g_ws.planes_cap, plane_bytes);
        if (g_ws.planes) cudaFree(g_ws.planes);
        g_ws.planes = nullptr; g_ws.planes_cap = 0;
        SKB_CUDA_CHECK(cudaMalloc(&g_ws.planes, plane_bytes));
        g_ws.planes_cap = plane_bytes;
    }
    if (tmp_bytes > g_ws.tmp_cap) {
        if (getenv("SKB_TRACE_ALLOC")) fprintf(stderr, "skb: scoring scratch grows %zu -> %zu bytes\n", g_ws.tmp_cap, tmp_bytes);
        if (g_ws.tmp) cudaFree(g_ws.tmp);
        g_ws.tmp = nullptr; g_ws.tmp_cap = 0;
        SKB_CUDA_CHECK(cudaMalloc(&g_ws.tmp, tmp_bytes));
        g_ws.tmp_cap = tmp_bytes;
    }
    return SKB_OK;
}

static int packed_alloc(PackedOp* op, int rows, int D) {
    op->rows = rows; op->D = D;
    op->Dp = (D + kScKChunk - 1) / kScKChunk * kScKChunk;
    op->rows_pad = (rows + 127) / 128 * 128;
    const size_t halves = (size_t)op->Dp * op->rows_pad;
    SKB_CUDA_CHECK(cudaMalloc(&op->hi, 2 * halves * sizeof(uint16_t)));
    op->lo = op->hi + halves;
    SKB_CUDA_CHECK(cudaMalloc(&op->stats, 2 * sizeof(unsigned) + sizeof(int)));
    op->exp = reinterpret_cast<int*>(op->stats + 2);
    return SKB_OK;
}

void packed_free(PackedOp* op) {
    cudaFree(op->hi);
    cudaFree(op->stats);
    *op = PackedOp();
}

// scale, split into fp16 hi / lo and lay out as 128-row tiles of chunk planes (buffers of the operands already sized);
// one or two operands (same D) per pair of launches
static int packed_fill(const float* X0, PackedOp* op0, const float* X1, PackedOp* op1, cudaStream_t st) {
    const int n_ops = op1 ? 2 : 1;
    int rc = ws_ensure(0, 0);
    if (rc) return rc;
    AbsmaxArgs aa;
    PackArgs pa;
    PackedOp* ops[2] = {op0, op1};
    const float* Xs[2] = {X0, X1};
    int max_rows = 0, max_tiles = 0;
    for (int i = 0; i < 2; ++i) {
        PackedOp* o = ops[i < n_ops ? i : 0];
        aa.X[i] = pa.X[i] = Xs[i < n_ops ? i : 0];
        aa.rows[i] = pa.rows[i] = o->rows;
        aa.stats[i] = o->stats;
        aa.partial[i] = g_ws.partial + (size_t)i * kAbsmaxMaxCtas;
        aa.ticket[i] = g_ws.ticket + i;
        pa.stats[i] = o->stats;
        pa.rows_pad[i] = o->rows_pad; pa.exp_out[i] = o->exp; pa.hi[i] = o->hi; pa.lo[i] = o->lo;
        if (i < n_ops) {
            max_rows = std::max(max_rows, o->rows);
            max_tiles = std::max(max_tiles, o->rows_pad / 128);
        }
    }
    SKB_CUDA_CHECK(launch_kernel(true, absmax_kernel, dim3(std::max(1, std::min((max_rows + kAbsmaxWarps - 1) / kAbsmaxWarps, kAbsmaxMaxCtas)), n_ops),
                                 dim3(kAbsmaxWarps * 32), 0, st, aa, op0->D));
    SKB_CUDA_CHECK(launch_kernel(true, pack_split_kernel, dim3((unsigned)std::max(1, max_tiles), op0->Dp / 64, n_ops), dim3(256), 0, st, pa, op0->D,
                                 op0->Dp));
    return SKB_OK;
}

int packed_create(const float* X_dev, int rows, int D, PackedOp* op, cudaStream_t st) {
    int rc = packed_alloc(op, rows, D);
    if (rc) return rc;
    return packed_fill(X_dev, op, nullptr, nullptr, st);
}

// pre-size the workspace of gemm_nt_split for A operands of up to M rows x K columns (skb_xtractor_reserve)
int gemm_workspace_reserve(int M, int K) {
    const int Dp = (K + kScKChunk - 1) / kScKChunk * kScKChunk, Mp = (M + 127) / 128 * 128;
    return ws_ensure(2 * (size_t)Dp * Mp * sizeof(uint16_t), 0);
}

// workspace-backed operand view (slot 0 / 1 of the plane buffer, stats slots in g_ws.stats)
static void ws_operand(PackedOp* op, int rows, int D, int slot, size_t offset_halves) {
    op->rows = rows; op->D = D;
    op->Dp = (D + kScKChunk - 1) / kScKChunk * kScKChunk;
    op->rows_pad = (rows + 127) / 128 * 128;
    op->hi = g_ws.planes + offset_halves;
    op->lo = op->hi + (size_t)op->Dp * op->rows_pad;
    op->stats = g_ws.stats + 3 * slot;
    op->exp = reinterpret_cast<int*>(op->stats + 2);
}

// Shared memory is sized for the forced pass count, or for the larger of the two layouts when the device decides.
template <bool STREAM_A, int MODE, int KC = 64>
static int launch_score(const ScoreParams& p, cudaStream_t st) {
    static PerDeviceOnce configured;
    const size_t smem1 = ScoreSmem<1, STREAM_A, KC>::total(p.topk_k), smem3 = ScoreSmem<3, STREAM_A>::total(p.topk_k);
    const size_t smem = p.passes_req == 1 ? smem1 : (p.passes_req == 3 ? smem3 : std::max(smem1, smem3));
    const int grid = std::min((p.Ne_pad / 128) * p.n_ntiles, kNumSMs);
    if (smem > 227 * 1024) {
        set_last_error(__FILE__, __LINE__, "score_gemm: the stage ring does not fit in shared memory");
        return SKB_ERR_ARG;
    }
    if (configured.first()) {
        SKB_CUDA_CHECK(cudaFuncSetAttribute(score_gemm_kernel<STREAM_A, MODE, KC>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    }
    SKB_CUDA_CHECK(launch_kernel(true, score_gemm_kernel<STREAM_A, MODE, KC>, dim3(grid), dim3(ScoreSmem<1, STREAM_A>::kThreads), smem, st, p));
    return SKB_OK;
}

// out = acc * (ra_i + ca_j + a0) + rq_scale * (r_i + q_j) + c0 on two packed operands
int gemm_packed(const PackedOp& E, const PackedOp& T, const float* ra, const float* ca, float a0, const float* r, const float* q,
                float c0, float rq_scale, float abs_alpha_for_auto, int passes, int out_mode, void* out, long long ld_out,
                cudaStream_t st, const TrialTables* trials, const TopkLists* topk = nullptr) {
    if (E.Dp != T.Dp || !out || (out_mode < 3 && ld_out < T.rows) || (passes != 0 && passes != 1 && passes != 3) || out_mode < 0 ||
        out_mode > 4 || (out_mode == 3 && (trials == nullptr || trials->Ne != E.rows || trials->Nt != T.rows || ca != nullptr)) ||
        (out_mode == 4 && (topk == nullptr || topk->k < 1 || topk->k > 32 || ca != nullptr))) {
        set_last_error(__FILE__, __LINE__, "gemm_packed: bad arguments");
        return SKB_ERR_ARG;
    }
    int rc = ws_ensure(0, 0);
    if (rc) return rc;
    ScoreParams p;
    p.Ehi = E.hi; p.Elo = E.lo; p.Thi = T.hi; p.Tlo = T.lo;
    p.Ne = E.rows; p.Nt = T.rows; p.Ne_pad = E.rows_pad; p.Dp = E.Dp; p.D = E.D;
    p.expE = E.exp; p.expT = T.exp; p.statsE = E.stats; p.statsT = T.stats;
    p.abs_alpha = abs_alpha_for_auto; p.passes_req = passes;
    p.ra = ra; p.ca = ca; p.r = r; p.q = q; p.a0 = a0; p.c0 = c0; p.rq_scale = rq_scale;
    p.mul_scaled = 1;
    p.out = out; p.ld_out = ld_out; p.out_mode = out_mode;
    p.mask_words = trials ? trials->words : nullptr;
    p.word_off = trials ? trials->offsets : nullptr;
    p.mask_ld = trials ? trials->ld : 0;
    p.topk_k = topk ? topk->k : 0;
    p.topk_segs = topk ? topk->segs : 0;
    p.n_ntiles = T.rows_pad / 128;
    // Large K (dense layers of the pooling / head) streams both operands; K <= 256 keeps the E panel resident, in
    // 128-wide ring stages whenever the padded K allows (see ScoreSmem)
    if (E.Dp > 256) {
        if (out_mode == 3 || out_mode == 4) {
            set_last_error(__FILE__, __LINE__, out_mode == 3 ? "trial-list mode supports embeddings of up to 256 dimensions"
                                                             : "top-k epilogue supports embeddings of up to 256 dimensions");
            return SKB_ERR_ARG;
        }
        return launch_score<true, kEpiMatrix>(p, st);
    }
    const bool wide = E.Dp % 128 == 0;
    if (out_mode == 3) return wide ? launch_score<false, kEpiTrials, 128>(p, st) : launch_score<false, kEpiTrials, 64>(p, st);
    if (out_mode == 4) return wide ? launch_score<false, kEpiTopk, 128>(p, st) : launch_score<false, kEpiTopk, 64>(p, st);
    return wide ? launch_score<false, kEpiMatrix, 128>(p, st) : launch_score<false, kEpiMatrix, 64>(p, st);
}

// C[m][n] = sum_k A[m][k] * W[n][k] + bias[n] with fp32-class accuracy (split fp16 passes): the dense layers of the
// attentive pooling and the embedding / margin heads.  W is packed once at model-build time.
int gemm_nt_split(const float* A_dev, int M, int K, const PackedOp& W, const float* bias, float alpha, float* C, int ldc,
                  cudaStream_t st) {
    if (K != W.D) {
        set_last_error(__FILE__, __LINE__, "gemm_nt_split: K mismatch");
        return SKB_ERR_ARG;
    }
    const int Dp = W.Dp, Mp = (M + 127) / 128 * 128;
    int rc = ws_ensure(2 * (size_t)Dp * Mp * sizeof(uint16_t), 0);
    if (rc) return rc;
    PackedOp a;
    ws_operand(&a, M, K, 0, 0);
    if ((rc = packed_fill(A_dev, &a, nullptr, nullptr, st))) return rc;
    return gemm_packed(a, W, nullptr, nullptr, alpha, nullptr, bias, 0.f, 1.f, 1.f, 3, 0, C, ldc, st, nullptr);
}

// An operand whose hi planes the caller fills itself (16-bit activations gathered straight into the packed layout):
// everything zeroed, so lo = 0 and the scale exponent is 0.
int packed_alloc_zero(PackedOp* op, int rows, int D, cudaStream_t st) {
    int rc = packed_alloc(op, rows, D);
    if (rc) return rc;
    SKB_CUDA_CHECK(cudaMemsetAsync(op->hi, 0, 2 * (size_t)op->Dp * op->rows_pad * sizeof(uint16_t), st));
    SKB_CUDA_CHECK(cudaMemsetAsync(op->stats, 0, 2 * sizeof(unsigned) + sizeof(int), st));
    return SKB_OK;
}

int gemm_packed_a(const PackedOp& A, const PackedOp& W, const float* bias, float alpha, float* C, int ldc, cudaStream_t st) {
    return gemm_packed(A, W, nullptr, nullptr, alpha, nullptr, bias, 0.f, 1.f, 1.f, 3, 0, C, ldc, st, nullptr);
}

// out = acc * (ra_i + ca_j + a0) + rq_scale * (r_i + q_j) + c0 from fp32 row-major operands
static int score_gemm_general(const float* E, const float* T, int Ne, int Nt, int D, const float* ra, const float* ca, float a0,
                              const float* r, const float* q, float c0, float rq_scale, float abs_alpha_for_auto, int passes, int out_mode,
                              void* out, long long ld_out, size_t tmp_bytes, cudaStream_t st, const TrialTables* trials = nullptr) {
    if (!E || !T || !out || Ne <= 0 || Nt <= 0 || D <= 0 || (out_mode != 3 && ld_out < Nt)) {
        set_last_error(__FILE__, __LINE__, "score_gemm: bad arguments");
        return SKB_ERR_ARG;
    }
    const int Dp = (D + kScKChunk - 1) / kScKChunk * kScKChunk;
    const size_t eh = (size_t)Dp * ((Ne + 127) / 128 * 128), th = (size_t)Dp * ((Nt + 127) / 128 * 128);
    int rc = ws_ensure(2 * (eh + th) * sizeof(uint16_t), tmp_bytes);
    if (rc) return rc;
    PackedOp e, t;
    ws_operand(&e, Ne, D, 0, 0);
    ws_operand(&t, Nt, D, 1, 2 * eh);
    if ((rc = packed_fill(E, &e, T, &t, st))) return rc;
    return gemm_packed(e, t, ra, ca, a0, r, q, c0, rq_scale, abs_alpha_for_auto, passes, out_mode, out, ld_out, st, trials);
}

// ----------------------------------------------------------------------------- trial index (trial-list mode)
// mask (Ne, Nt) bytes -> bit words + exclusive row-major prefix counts.  One warp per row: 128 mask bytes per step (a
// 32-bit load per lane), ballots assemble four words, the in-row offsets follow from a running popcount.
__global__ void trial_words_kernel(const uint8_t* __restrict__ mask, int Ne, int Nt, long long ld, uint32_t* __restrict__ words,
                                   uint32_t* __restrict__ offs, int mask_ld, uint32_t* __restrict__ row_total) {
    const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (row >= Ne) return;
    const uint8_t* m = mask + (size_t)row * ld;
    uint32_t running = 0;
    for (int w0 = 0; w0 < mask_ld; w0 += 32) {
        // lane handles word w0 + lane: its 32 mask bytes
        const int w = w0 + lane;
        uint32_t word = 0u;
        if (w < mask_ld) {
            const int c0 = w * 32;
#pragma unroll 4
            for (int j = 0; j < 32; ++j) {
                const int c = c0 + j;
                if (c < Nt && m[c]) word |= 1u << j;
            }
        }
        const uint32_t cnt = __popc(word);
        uint32_t incl = cnt;                       // warp inclusive scan of the 32 word counts
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t v = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += v;
        }
        if (w < mask_ld) {
            words[(size_t)row * mask_ld + w] = word;
            offs[(size_t)row * mask_ld + w] = running + incl - cnt;
        }
        running += __shfl_sync(0xffffffffu, incl, 31);
    }
    if (lane == 0) row_total[row] = running;
}

// exclusive scan of the row totals (one CTA; Ne is at most a few 10^5) -> row_base; total -> *n_trials
__global__ void __launch_bounds__(1024) trial_rowscan_kernel(const uint32_t* __restrict__ row_total, int Ne, uint32_t* __restrict__ row_base,
                                                             unsigned long long* __restrict__ n_trials) {
    __shared__ unsigned long long warp_tot[32];
    __shared__ unsigned long long carry;
    if (threadIdx.x == 0) carry = 0ull;
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int base = 0; base < Ne; base += 1024) {
        const int i = base + threadIdx.x;
        const unsigned long long v = i < Ne ? row_total[i] : 0ull;
        unsigned long long incl = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned long long u = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += u;
        }
        if (lane == 31) warp_tot[warp] = incl;
        __syncthreads();
        unsigned long long before = carry;
        for (int k = 0; k < warp; ++k) before += warp_tot[k];
        if (i < Ne) row_base[i] = (uint32_t)(before + incl - v);
        __syncthreads();
        if (threadIdx.x == 1023) carry = before + incl;
        __syncthreads();
    }
    if (threadIdx.x == 0) *n_trials = carry;
}

__global__ void trial_addbase_kernel(uint32_t* __restrict__ offs, const uint32_t* __restrict__ row_base, long long n, int mask_ld) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) offs[i] += row_base[i / mask_ld];
}

// ----------------------------------------------------------------------------- as-norm: top-k statistics per row
// Block-wide radix select (blockDim.x == 256, every thread calls it once per launch): the k-th largest of the C keys
// key_at(0 .. C-1) (.x) and how many of the keys equal to it are among the k largest (.y).  Four 8-bit passes.
template <class KeyAt>
__device__ uint2 radix_select_kth(KeyAt key_at, int C, unsigned k) {
    __shared__ unsigned hist[256];
    __shared__ unsigned sel_prefix, sel_remaining;
    if (threadIdx.x == 0) { sel_prefix = 0; sel_remaining = k; }
    __syncthreads();
    for (int shift = 24; shift >= 0; shift -= 8) {
        hist[threadIdx.x] = 0;
        __syncthreads();
        const unsigned prefix = sel_prefix;
        const unsigned mask = shift == 24 ? 0u : (0xffffffffu << (shift + 8));
        for (int i = threadIdx.x; i < C; i += blockDim.x) {
            const unsigned key = key_at(i);
            if ((key & mask) == (prefix & mask)) atomicAdd(&hist[(key >> shift) & 255], 1u);
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            unsigned rem = sel_remaining;
            int b = 255;
            for (; b > 0; --b) {
                if (hist[b] >= rem) break;
                rem -= hist[b];
            }
            sel_prefix = prefix | ((unsigned)b << shift);
            sel_remaining = rem;          // how many of the keys equal to the final threshold are taken
        }
        __syncthreads();
    }
    return make_uint2(sel_prefix, sel_remaining);
}

// One CTA per row: radix-select the k-th largest score, then mean and unbiased std of the top k
// (torch.topk + mean + std, sidekit/score_normalization.py:131-133).  Ties at the threshold are
// counted exactly k - (#greater) times, like a sort would.
__global__ void __launch_bounds__(256) topk_stats_kernel(const float* __restrict__ S, int C, long long ld, int k,
                                                         float* __restrict__ mean_out, float* __restrict__ std_out) {
    extern __shared__ unsigned keys[];
    __shared__ double red[2][8];
    const float* row = S + (size_t)blockIdx.x * ld;
    for (int i = threadIdx.x; i < C; i += blockDim.x) keys[i] = f2key(row[i]);
    __syncthreads();
    const uint2 sel = radix_select_kth([&](int i) { return keys[i]; }, C, (unsigned)k);
    const unsigned thr = sel.x;
    const unsigned n_thr = sel.y;
    const float thr_f = key2f(thr);
    // pass 1: mean
    double s = 0.0;
    for (int i = threadIdx.x; i < C; i += blockDim.x)
        if (keys[i] > thr) s += (double)key2f(keys[i]);
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if ((threadIdx.x & 31) == 0) red[0][threadIdx.x >> 5] = s;
    __syncthreads();
    double tot = 0.0;
    for (int i = 0; i < 8; ++i) tot += red[0][i];
    const double mean = (tot + (double)n_thr * thr_f) / k;
    double v = 0.0;
    for (int i = threadIdx.x; i < C; i += blockDim.x)
        if (keys[i] > thr) {
            const double d = (double)key2f(keys[i]) - mean;
            v += d * d;
        }
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31) == 0) red[1][threadIdx.x >> 5] = v;
    __syncthreads();
    if (threadIdx.x == 0) {
        double vt = 0.0;
        for (int i = 0; i < 8; ++i) vt += red[1][i];
        const double d = (double)thr_f - mean;
        vt += (double)n_thr * d * d;
        mean_out[blockIdx.x] = (float)mean;
        std_out[blockIdx.x] = (float)sqrt(vt / (k - 1));
    }
}

// ----------------------------------------------------------------------------- top-k columns per row
// Fused path (k <= kTopkFusedMax, D <= 256): the GEMM's top-k epilogue leaves partial lists; one warp per row merges the
// row's segments (topk_panel_segs of its panel, k keys each, padded with key 0) into the final k, descending.
constexpr int kTopkFusedMax = 32;
constexpr int kTopkMax = 1024;
__global__ void __launch_bounds__(256) topk_merge_kernel(const unsigned long long* __restrict__ lists, int Ne, int k, int segs,
                                                         int n_ntiles, int tiles, int grid, float* __restrict__ values,
                                                         int64_t* __restrict__ indices) {
    pdl_wait();
    const int row = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (row >= Ne) return;
    const int n = topk_panel_segs(row >> 7, n_ntiles, tiles, grid) * k;
    const unsigned long long* __restrict__ L = lists + (size_t)row * segs * k;
    // k rounds of a warp arg-max below the previous pick (the non-zero keys of a row are distinct: one per column)
    unsigned long long last = ~0ull;
    for (int r = 0; r < k; ++r) {
        unsigned long long best = 0ull;
        for (int i = lane; i < n; i += 32) {
            const unsigned long long x = __ldg(L + i);
            if (x < last && x > best) best = x;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) best = max(best, __shfl_xor_sync(0xffffffffu, best, o));
        last = best;
        if (lane == (r & 31)) {
            values[(size_t)row * k + r] = key2f((unsigned)(best >> 32));
            indices[(size_t)row * k + r] = (int64_t)(int)~(unsigned)best;   // padding (key 0) -> -1
        }
    }
}

// Panel path (k > kTopkFusedMax or D > 256): one CTA per row of a float32 score panel.  Radix-select the k-th key, keep every
// key above it and the lowest-index ties at it (k survivors), sort them in shared memory in the same 64-bit order.
__global__ void __launch_bounds__(256) topk_select_kernel(const float* __restrict__ S, int C, long long ld, int k,
                                                          float* __restrict__ values, int64_t* __restrict__ indices) {
    extern __shared__ unsigned long long cand[];          // [kp], kp = next power of two >= k
    __shared__ unsigned n_greater, taken, w_cnt[8];
    const float* __restrict__ row = S + (size_t)blockIdx.x * ld;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint2 sel = radix_select_kth([&](int i) { return f2key(__ldg(row + i)); }, C, (unsigned)k);
    const unsigned thr = sel.x, n_thr = sel.y;
    int kp = 1;
    while (kp < k) kp <<= 1;
    for (int i = threadIdx.x; i < kp; i += blockDim.x) cand[i] = 0ull;
    if (threadIdx.x == 0) { n_greater = 0u; taken = 0u; }
    __syncthreads();
    for (int i = threadIdx.x; i < C; i += blockDim.x) {
        const unsigned key = f2key(__ldg(row + i));
        if (key > thr) cand[atomicAdd(&n_greater, 1u)] = ((unsigned long long)key << 32) | (unsigned)~i;
    }
    __syncthreads();
    const unsigned g = n_greater;                         // == k - n_thr
    // the n_thr ties at the threshold with the lowest column indices: a block-wide ordered scan, 256 columns per step
    for (int base = 0; base < C && taken < n_thr; base += blockDim.x) {
        const int i = base + threadIdx.x;
        const bool eq = i < C && f2key(__ldg(row + i)) == thr;
        const unsigned ball = __ballot_sync(0xffffffffu, eq);
        if (lane == 0) w_cnt[warp] = __popc(ball);
        __syncthreads();
        unsigned pos = taken + __popc(ball & ((1u << lane) - 1u));
        for (int w = 0; w < warp; ++w) pos += w_cnt[w];
        if (eq && pos < n_thr) cand[g + pos] = ((unsigned long long)thr << 32) | (unsigned)~i;
        __syncthreads();
        if (threadIdx.x == 0)
            for (int w = 0; w < 8; ++w) taken += w_cnt[w];
        __syncthreads();
    }
    // bitonic sort, descending
    for (int size = 2; size <= kp; size <<= 1)
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            for (int i = threadIdx.x; i < kp; i += blockDim.x) {
                const int j = i ^ stride;
                if (j > i) {
                    const unsigned long long a = cand[i], b = cand[j];
                    if ((i & size) == 0 ? a < b : a > b) { cand[i] = b; cand[j] = a; }
                }
            }
            __syncthreads();
        }
    for (int r = threadIdx.x; r < k; r += blockDim.x) {
        const unsigned long long x = cand[r];
        values[(size_t)blockIdx.x * k + r] = key2f((unsigned)(x >> 32));
        indices[(size_t)blockIdx.x * k + r] = (int64_t)(int)~(unsigned)x;
    }
}

// The k best columns of every row of S = acc * a0 + rq_scale * (r_i + q_j) + c0 for two packed operands.  The operands are
// packed once for the whole call, so the scale exponents and the pass decision are those of the matching score_matrix call
// and every selected value is its matrix entry bit for bit.  1 <= k <= min(T.rows, kTopkMax) is checked by the caller.
static int score_topk_packed(const PackedOp& e, const PackedOp& t, const float* r, const float* q, float a0, float c0, float rq_scale,
                             float abs_alpha, int passes, int k, float* values, int64_t* indices, cudaStream_t st) {
    int rc;
    if (k <= kTopkFusedMax && e.Dp <= 256) {
        // the partial-list scratch [Ne][segs][k] is sized from the partition score_gemm_body uses (one row panel per item)
        const int n_panels = e.rows_pad / 128, n_ntiles = t.rows_pad / 128;
        const int tiles = n_panels * n_ntiles, grid = std::min(tiles, kNumSMs);
        int segs = 0;
        for (int P = 0; P < n_panels; ++P) segs = std::max(segs, topk_panel_segs(P, n_ntiles, tiles, grid));
        if ((rc = ws_ensure(0, (size_t)e.rows * segs * k * sizeof(unsigned long long)))) return rc;
        TopkLists tl{reinterpret_cast<unsigned long long*>(g_ws.tmp), k, segs};
        if ((rc = gemm_packed(e, t, nullptr, nullptr, a0, r, q, c0, rq_scale, abs_alpha, passes, 4, tl.keys, 0, st, nullptr, &tl))) return rc;
        SKB_CUDA_CHECK(launch_kernel(true, topk_merge_kernel, dim3((unsigned)((e.rows + 7) / 8)), dim3(256), 0, st,
                                     (const unsigned long long*)tl.keys, e.rows, k, segs, n_ntiles, tiles, grid, values, indices));
        return SKB_OK;
    }
    // Row panels of the score matrix through a bounded float32 scratch (<= 1 GB, at least one 128-row tile), each followed by
    // the per-row select.  A panel is a view of the packed E (whole 128-row tiles): same statistics, same arithmetic.
    const long long ld = (t.rows + 3) / 4 * 4;
    constexpr long long kPanelBytes = 1ll << 30;
    const int rows = (int)std::min<long long>(e.rows_pad, std::max<long long>(128, kPanelBytes / (ld * 4) / 128 * 128));
    if ((rc = ws_ensure(0, (size_t)rows * ld * sizeof(float)))) return rc;
    int kp = 1;
    while (kp < k) kp <<= 1;
    for (int r0 = 0; r0 < e.rows; r0 += rows) {
        PackedOp v = e;
        v.rows = std::min(rows, e.rows - r0);
        v.rows_pad = (v.rows + 127) / 128 * 128;
        v.hi = e.hi + (size_t)r0 * e.Dp;
        v.lo = e.lo + (size_t)r0 * e.Dp;
        if ((rc = gemm_packed(v, t, nullptr, nullptr, a0, r ? r + r0 : nullptr, q, c0, rq_scale, abs_alpha, passes, 0, g_ws.tmp, ld, st,
                              nullptr)))
            return rc;
        SKB_CUDA_CHECK(launch_kernel(false, topk_select_kernel, dim3(v.rows), dim3(256), kp * sizeof(unsigned long long), st, g_ws.tmp, t.rows,
                                     ld, k, values + (size_t)r0 * k, indices + (size_t)r0 * k));
    }
    return SKB_OK;
}

static int topk_check_args(int Ne, int Nt, int k, int passes) {
    if (Ne < 1 || Nt < 1 || (passes != 0 && passes != 1 && passes != 3)) {
        set_last_error(__FILE__, __LINE__, "score_gemm_topk: bad arguments");
        return SKB_ERR_ARG;
    }
    if (k < 1 || k > Nt || k > kTopkMax) {
        set_last_error(__FILE__, __LINE__, "score_gemm_topk: need 1 <= k <= min(Nt, 1024)");
        return SKB_ERR_ARG;
    }
    return SKB_OK;
}

// ra_i = 0.5 / std_i,  r_i = -0.5 * mean_i / std_i   (the symmetric as-norm as acc*(ra_i+ra_j) + (r_i+r_j))
__global__ void asnorm_terms_kernel(const float* mean, const float* sd, int N, float* ra, float* r) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N) return;
    ra[i] = 0.5f / sd[i];
    r[i] = -0.5f * mean[i] / sd[i];
}

// x - mu (row-wise); rowterm_i = 0.5 * sum_j tmp[i][j] * xc[i][j]
__global__ void center_kernel(const float* __restrict__ X, const float* __restrict__ mu, int N, int D, float* __restrict__ out) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (long long)N * D) return;
    out[i] = X[i] - (mu ? mu[i % D] : 0.f);
}
__global__ void half_rowdot_kernel(const float* __restrict__ A, const float* __restrict__ B, int N, int D, float* __restrict__ out) {
    const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (row >= N) return;
    const int lane = threadIdx.x & 31;
    float s = 0.f;
    for (int k = lane; k < D; k += 32) s = fmaf(A[(size_t)row * D + k], B[(size_t)row * D + k], s);
    s = warp_sum(s);
    if (lane == 0) out[row] = 0.5f * s;
}

// float32 -> float64 on the way to the host (the reference's PLDA scorers return float64; the GEMM keeps float32)
__global__ void widen_kernel(const float* __restrict__ src, double* __restrict__ dst, long long n) {
    const long long i = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * 4;
    if (i + 4 <= n && (reinterpret_cast<uintptr_t>(src + i) & 15) == 0) {
        const float4 v = __ldcs(reinterpret_cast<const float4*>(src + i));
        __stcs(reinterpret_cast<double2*>(dst + i), make_double2((double)v.x, (double)v.y));
        __stcs(reinterpret_cast<double2*>(dst + i) + 1, make_double2((double)v.z, (double)v.w));
    } else {
        for (long long k = i; k < n && k < i + 4; ++k) dst[k] = (double)src[k];
    }
}

// ----------------------------------------------------------------------------- pair-list scoring
// One score per (rows[p], cols[p]) trial: a gather of two rows and a D-term dot product, about 8 bytes read per 2 FLOP, so
// the kernel is bound by the row loads and the tensor core has nothing to add.  kPairLanes lanes own one trial: lane l sums
// the products of columns l, l + kPairLanes, ... (float4 units when VEC) in ascending order with float32 FMAs, then a fixed
// xor butterfly over the group adds the partials.  So the bits of a score depend on D and the two rows only, not on the
// trial's position, the list length or the grid.  Any D works (the loop has no tile); VEC needs D % 4 == 0 and 16-byte
// aligned bases.  An index outside [0, Ne) / [0, Nt) is never dereferenced: its trial gets NaN.
constexpr int kPairLanes = 8;
constexpr int kPairThreads = 256;
constexpr int kPairsPerCta = kPairThreads / kPairLanes;
struct PairArgs {
    const float* E; const float* T; int Ne, Nt, D;
    const int32_t* rows; const int32_t* cols; long long n;
    const float* rowterm; const float* colterm; float cst, alpha;
    const float* mean_e; const float* std_e; const float* mean_t; const float* std_t;    // all NULL: no as-norm
    float* out;
};

template <bool VEC>
__global__ void __launch_bounds__(kPairThreads) score_pairs_kernel(const PairArgs a) {
    pdl_wait();
    const int sub = threadIdx.x & (kPairLanes - 1);
    const long long p = (long long)blockIdx.x * kPairsPerCta + threadIdx.x / kPairLanes;
    int i = -1, j = -1;
    if (p < a.n) { i = __ldg(a.rows + p); j = __ldg(a.cols + p); }
    const bool ok = p < a.n && (unsigned)i < (unsigned)a.Ne && (unsigned)j < (unsigned)a.Nt;
    float acc = 0.f;
    if (ok) {
        const float* __restrict__ e = a.E + (size_t)i * a.D;
        const float* __restrict__ t = a.T + (size_t)j * a.D;
        if (VEC) {
            const float4* __restrict__ e4 = reinterpret_cast<const float4*>(e);
            const float4* __restrict__ t4 = reinterpret_cast<const float4*>(t);
            const int n4 = a.D >> 2;
            int k = sub;
            for (; k + 3 * kPairLanes < n4; k += 4 * kPairLanes) {          // four float4 of each row in flight per lane
                float4 x[4], y[4];
#pragma unroll
                for (int u = 0; u < 4; ++u) { x[u] = __ldg(e4 + k + u * kPairLanes); y[u] = __ldg(t4 + k + u * kPairLanes); }
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    acc = fmaf(x[u].x, y[u].x, acc); acc = fmaf(x[u].y, y[u].y, acc);
                    acc = fmaf(x[u].z, y[u].z, acc); acc = fmaf(x[u].w, y[u].w, acc);
                }
            }
            for (; k < n4; k += kPairLanes) {
                const float4 x = __ldg(e4 + k), y = __ldg(t4 + k);
                acc = fmaf(x.x, y.x, acc); acc = fmaf(x.y, y.y, acc); acc = fmaf(x.z, y.z, acc); acc = fmaf(x.w, y.w, acc);
            }
        } else {
            for (int k = sub; k < a.D; k += kPairLanes) acc = fmaf(__ldg(e + k), __ldg(t + k), acc);
        }
    }
#pragma unroll
    for (int o = kPairLanes / 2; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if (p >= a.n || sub != 0) return;
    if (!ok) {
        a.out[p] = __int_as_float(0x7fc00000);
        return;
    }
    // the score_matrix convention: alpha * (rowterm_i + colterm_j + cst) + alpha * dot
    const float terms = (a.rowterm ? __ldg(a.rowterm + i) : 0.f) + (a.colterm ? __ldg(a.colterm + j) : 0.f) + a.cst;
    float s = fmaf(a.alpha, acc, a.alpha * terms);
    if (a.mean_e)      // symmetric as-norm, sidekit/score_normalization.py:135-138
        s = 0.5f * (s - __ldg(a.mean_e + i)) / __ldg(a.std_e + i) + 0.5f * (s - __ldg(a.mean_t + j)) / __ldg(a.std_t + j);
    a.out[p] = s;
}

}  // namespace skb

using namespace skb;

extern "C" {

int skb_quadratic_prepare(const float* X_dev, const float* mu_dev, const float* PsiT_dev, const float* Phi_dev, int N, int D,
                          float* Xout_dev, float* rowterm_dev, void* stream) {
    if (!X_dev || !Phi_dev || !Xout_dev || !rowterm_dev || N <= 0 || D <= 0) {
        set_last_error(__FILE__, __LINE__, "quadratic_prepare: bad arguments");
        return SKB_ERR_ARG;
    }
    cudaStream_t st = (cudaStream_t)stream;
    const size_t nd = (size_t)N * D;
    int rc = ws_ensure(0, 2 * nd * sizeof(float));
    if (rc) return rc;
    float* xc = g_ws.tmp;
    float* tmp = g_ws.tmp + nd;
    SKB_CUDA_CHECK(launch_kernel(false, center_kernel, dim3((unsigned)((nd + 255) / 256)), dim3(256), 0, st, X_dev, mu_dev, N, D, xc));
    // tmp = xc . Phi  (Phi symmetric, so rows of Phi serve as the K-major "T" operand)
    rc = score_gemm_general(xc, Phi_dev, N, D, D, nullptr, nullptr, 1.f, nullptr, nullptr, 0.f, 1.f, 1.f, 3, 0, tmp, D,
                            2 * nd * sizeof(float), st);
    if (rc) return rc;
    SKB_CUDA_CHECK(launch_kernel(false, half_rowdot_kernel, dim3((N + 7) / 8), dim3(256), 0, st, tmp, xc, N, D, rowterm_dev));
    if (PsiT_dev) {
        rc = score_gemm_general(xc, PsiT_dev, N, D, D, nullptr, nullptr, 1.f, nullptr, nullptr, 0.f, 1.f, 1.f, 3, 0, Xout_dev, D,
                                2 * nd * sizeof(float), st);
        if (rc) return rc;
    } else {
        SKB_CUDA_CHECK(cudaMemcpyAsync(Xout_dev, xc, nd * sizeof(float), cudaMemcpyDeviceToDevice, st));
    }
    return SKB_OK;
}

int skb_score_gemm(const float* E_dev, const float* T_dev, int Ne, int Nt, int D, const float* rowterm_dev,
                   const float* colterm_dev, double cst, double alpha, int passes, int out_dtype, void* out_dev,
                   int64_t ld_out, void* stream) {
    return score_gemm_general(E_dev, T_dev, Ne, Nt, D, nullptr, nullptr, (float)alpha, rowterm_dev, colterm_dev,
                              (float)(alpha * cst), (float)alpha, (float)fabs(alpha), passes, out_dtype, out_dev, ld_out, 0,
                              (cudaStream_t)stream);
}

// ---- a test-side operand packed ONCE and scored against many enrol panels (multi-GPU row panels, repeated calls)
struct skb_packed { skb::PackedOp op; int device; };

int skb_packed_create(const float* X_dev, int rows, int D, skb_packed_t** out, void* stream) {
    if (!X_dev || !out || rows <= 0 || D <= 0) {
        set_last_error(__FILE__, __LINE__, "packed_create: bad arguments");
        return SKB_ERR_ARG;
    }
    skb_packed* p = new skb_packed();
    p->device = current_device();
    int rc = packed_create(X_dev, rows, D, &p->op, (cudaStream_t)stream);
    if (rc) {
        packed_free(&p->op);
        delete p;
        return rc;
    }
    *out = p;
    return SKB_OK;
}

void skb_packed_destroy(skb_packed_t* p) {
    if (!p) return;
    packed_free(&p->op);
    delete p;
}

int skb_score_gemm_packed(const float* E_dev, int Ne, const skb_packed_t* T, const float* rowterm_dev, const float* colterm_dev,
                          double cst, double alpha, int passes, int out_dtype, void* out_dev, int64_t ld_out, void* stream) {
    if (!E_dev || !T || !out_dev || Ne <= 0 || ld_out < T->op.rows) {
        set_last_error(__FILE__, __LINE__, "score_gemm_packed: bad arguments");
        return SKB_ERR_ARG;
    }
    if (T->device != current_device()) {
        set_last_error(__FILE__, __LINE__, "score_gemm_packed: the packed operand lives on another CUDA device");
        return SKB_ERR_STATE;
    }
    cudaStream_t st = (cudaStream_t)stream;
    const int D = T->op.D, Dp = T->op.Dp;
    const size_t eh = (size_t)Dp * ((Ne + 127) / 128 * 128);
    int rc = ws_ensure(2 * eh * sizeof(uint16_t), 0);
    if (rc) return rc;
    PackedOp e;
    ws_operand(&e, Ne, D, 0, 0);
    if ((rc = packed_fill(E_dev, &e, nullptr, nullptr, st))) return rc;
    return gemm_packed(e, T->op, nullptr, nullptr, (float)alpha, rowterm_dev, colterm_dev, (float)(alpha * cst), (float)alpha,
                       (float)fabs(alpha), passes, out_dtype, out_dev, ld_out, st, nullptr);
}

struct skb_trial_index { uint32_t *words = nullptr, *offsets = nullptr, *row_total = nullptr, *row_base = nullptr;
                         unsigned long long* n_dev = nullptr; int Ne = 0, Nt = 0, ld = 0, device = 0; long long n_trials = 0; };

void skb_trial_index_destroy(skb_trial_index_t* t) {
    if (!t) return;
    cudaFree(t->words); cudaFree(t->offsets); cudaFree(t->row_total); cudaFree(t->row_base); cudaFree(t->n_dev);
    delete t;
}

int skb_trial_index_create(const uint8_t* mask_dev, int Ne, int Nt, int64_t ld_mask, skb_trial_index_t** out, int64_t* n_trials,
                           void* stream) {
    if (!mask_dev || !out || !n_trials || Ne <= 0 || Nt <= 0 || ld_mask < Nt) {
        set_last_error(__FILE__, __LINE__, "trial_index_create: bad arguments");
        return SKB_ERR_ARG;
    }
    cudaStream_t st = (cudaStream_t)stream;
    skb_trial_index* t = new skb_trial_index();
    t->Ne = Ne; t->Nt = Nt; t->ld = (Nt + 31) / 32; t->device = current_device();
    const size_t nw = (size_t)Ne * t->ld;
    unsigned long long total = 0;
    if (cudaMalloc(&t->words, nw * 4) != cudaSuccess || cudaMalloc(&t->offsets, nw * 4) != cudaSuccess ||
        cudaMalloc(&t->row_total, (size_t)Ne * 4) != cudaSuccess || cudaMalloc(&t->row_base, (size_t)Ne * 4) != cudaSuccess ||
        cudaMalloc(&t->n_dev, 8) != cudaSuccess) {
        set_last_error(__FILE__, __LINE__, cudaGetErrorString(cudaGetLastError()));
        skb_trial_index_destroy(t);
        return SKB_ERR_CUDA;
    }
    cudaError_t e = launch_kernel(false, trial_words_kernel, dim3((Ne + 7) / 8), dim3(256), 0, st, mask_dev, Ne, Nt, (long long)ld_mask,
                                  t->words, t->offsets, t->ld, t->row_total);
    if (e == cudaSuccess) e = launch_kernel(false, trial_rowscan_kernel, dim3(1), dim3(1024), 0, st, t->row_total, Ne, t->row_base, t->n_dev);
    if (e == cudaSuccess)
        e = launch_kernel(false, trial_addbase_kernel, dim3((unsigned)((nw + 255) / 256)), dim3(256), 0, st, t->offsets, t->row_base,
                          (long long)nw, t->ld);
    if (e == cudaSuccess) e = cudaMemcpyAsync(&total, t->n_dev, 8, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) {
        set_last_error(__FILE__, __LINE__, cudaGetErrorString(e));
        skb_trial_index_destroy(t);
        return SKB_ERR_CUDA;
    }
    if (total >= 0xffffffffull) {
        set_last_error(__FILE__, __LINE__, "trial_index_create: more than 2^32 - 1 trials");
        skb_trial_index_destroy(t);
        return SKB_ERR_ARG;
    }
    t->n_trials = (long long)total;
    *n_trials = (int64_t)total;
    *out = t;
    return SKB_OK;
}

int skb_score_gemm_trials(const float* E_dev, const float* T_dev, int Ne, int Nt, int D, const float* rowterm_dev,
                          const float* colterm_dev, double cst, double alpha, int passes, const skb_trial_index_t* trials,
                          float* out_trials_dev, void* stream) {
    if (!trials || trials->Ne != Ne || trials->Nt != Nt || !out_trials_dev) {
        set_last_error(__FILE__, __LINE__, "score_gemm_trials: the trial index does not match the operands");
        return SKB_ERR_ARG;
    }
    if (trials->device != current_device()) {
        set_last_error(__FILE__, __LINE__, "score_gemm_trials: the trial index lives on another CUDA device");
        return SKB_ERR_STATE;
    }
    TrialTables tt{trials->words, trials->offsets, trials->ld, Ne, Nt};
    return score_gemm_general(E_dev, T_dev, Ne, Nt, D, nullptr, nullptr, (float)alpha, rowterm_dev, colterm_dev, (float)(alpha * cst),
                              (float)alpha, (float)fabs(alpha), passes, 3, out_trials_dev, 0, 0, (cudaStream_t)stream, &tt);
}

int skb_score_gemm_trials_packed(const float* E_dev, int Ne, const skb_packed_t* T, const float* rowterm_dev, const float* colterm_dev,
                                 double cst, double alpha, int passes, const skb_trial_index_t* trials, float* out_trials_dev,
                                 void* stream) {
    if (!E_dev || !T || !trials || trials->Ne != Ne || trials->Nt != T->op.rows || !out_trials_dev || Ne <= 0) {
        set_last_error(__FILE__, __LINE__, "score_gemm_trials_packed: the trial index does not match the operands");
        return SKB_ERR_ARG;
    }
    if (trials->device != current_device() || T->device != current_device()) {
        set_last_error(__FILE__, __LINE__, "score_gemm_trials_packed: the trial index / packed operand lives on another CUDA device");
        return SKB_ERR_STATE;
    }
    cudaStream_t st = (cudaStream_t)stream;
    const int D = T->op.D, Dp = T->op.Dp;
    const size_t eh = (size_t)Dp * ((Ne + 127) / 128 * 128);
    int rc = ws_ensure(2 * eh * sizeof(uint16_t), 0);
    if (rc) return rc;
    PackedOp e;
    ws_operand(&e, Ne, D, 0, 0);
    if ((rc = packed_fill(E_dev, &e, nullptr, nullptr, st))) return rc;
    TrialTables tt{trials->words, trials->offsets, trials->ld, Ne, T->op.rows};
    return gemm_packed(e, T->op, nullptr, nullptr, (float)alpha, rowterm_dev, colterm_dev, (float)(alpha * cst), (float)alpha,
                       (float)fabs(alpha), passes, 3, out_trials_dev, 0, st, &tt);
}

int skb_score_gemm_topk(const float* E_dev, const float* T_dev, int Ne, int Nt, int D, const float* rowterm_dev,
                        const float* colterm_dev, double cst, double alpha, int passes, int k, float* values_dev, int64_t* indices_dev,
                        void* stream) {
    if (!E_dev || !T_dev || !values_dev || !indices_dev || D <= 0) {
        set_last_error(__FILE__, __LINE__, "score_gemm_topk: bad arguments");
        return SKB_ERR_ARG;
    }
    int rc = topk_check_args(Ne, Nt, k, passes);
    if (rc) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    const int Dp = (D + kScKChunk - 1) / kScKChunk * kScKChunk;
    const size_t eh = (size_t)Dp * ((Ne + 127) / 128 * 128), th = (size_t)Dp * ((Nt + 127) / 128 * 128);
    if ((rc = ws_ensure(2 * (eh + th) * sizeof(uint16_t), 0))) return rc;
    PackedOp e, t;
    ws_operand(&e, Ne, D, 0, 0);
    ws_operand(&t, Nt, D, 1, 2 * eh);
    if ((rc = packed_fill(E_dev, &e, T_dev, &t, st))) return rc;
    return score_topk_packed(e, t, rowterm_dev, colterm_dev, (float)alpha, (float)(alpha * cst), (float)alpha, (float)fabs(alpha), passes,
                             k, values_dev, indices_dev, st);
}

int skb_score_gemm_topk_packed(const float* E_dev, int Ne, const skb_packed_t* T, const float* rowterm_dev, const float* colterm_dev,
                               double cst, double alpha, int passes, int k, float* values_dev, int64_t* indices_dev, void* stream) {
    if (!E_dev || !T || !values_dev || !indices_dev) {
        set_last_error(__FILE__, __LINE__, "score_gemm_topk_packed: bad arguments");
        return SKB_ERR_ARG;
    }
    int rc = topk_check_args(Ne, T->op.rows, k, passes);
    if (rc) return rc;
    if (T->device != current_device()) {
        set_last_error(__FILE__, __LINE__, "score_gemm_topk_packed: the packed operand lives on another CUDA device");
        return SKB_ERR_STATE;
    }
    cudaStream_t st = (cudaStream_t)stream;
    const int D = T->op.D, Dp = T->op.Dp;
    const size_t eh = (size_t)Dp * ((Ne + 127) / 128 * 128);
    if ((rc = ws_ensure(2 * eh * sizeof(uint16_t), 0))) return rc;
    PackedOp e;
    ws_operand(&e, Ne, D, 0, 0);
    if ((rc = packed_fill(E_dev, &e, nullptr, nullptr, st))) return rc;
    return score_topk_packed(e, T->op, rowterm_dev, colterm_dev, (float)alpha, (float)(alpha * cst), (float)alpha, (float)fabs(alpha), passes,
                             k, values_dev, indices_dev, st);
}

#ifdef SKB_SCORE_TIMING
int skb_debug_score_timing(unsigned long long* out16) {
    SKB_CUDA_CHECK(cudaDeviceSynchronize());
    SKB_CUDA_CHECK(cudaMemcpyFromSymbol(out16, skb::g_score_t, 16 * sizeof(unsigned long long)));
    unsigned long long z[16] = {0};
    SKB_CUDA_CHECK(cudaMemcpyToSymbol(skb::g_score_t, z, sizeof(z)));
    return SKB_OK;
}
#endif

int skb_widen_f32_f64(const float* src_dev, double* dst_dev, int64_t n, void* stream) {
    if (!src_dev || !dst_dev || n < 0) {
        set_last_error(__FILE__, __LINE__, "widen: bad arguments");
        return SKB_ERR_ARG;
    }
    if (n == 0) return SKB_OK;
    SKB_CUDA_CHECK(launch_kernel(false, widen_kernel, dim3((unsigned)((n + 1023) / 1024)), dim3(256), 0, (cudaStream_t)stream, src_dev, dst_dev,
                                 (long long)n));
    return SKB_OK;
}

int skb_asnorm_stats(const float* X_dev, const float* cohort_dev, int N, int C, int D, int top_k, float* mean_dev,
                     float* std_dev, void* stream) {
    if (top_k < 2 || C < top_k || C * sizeof(unsigned) > 200 * 1024) {
        set_last_error(__FILE__, __LINE__, "asnorm_stats: need 2 <= top_k <= C <= 51200");
        return SKB_ERR_ARG;
    }
    cudaStream_t st = (cudaStream_t)stream;
    const long long ld = (C + 3) / 4 * 4;
    // The N x C cohort score matrix never exists as a whole: the rows go through a bounded scratch panel (at most
    // kAsnormChunkRows x C scores, 473 MB at C = 7205) -- GEMM of the panel, radix-select statistics of its rows, next
    // panel -- so a million embeddings need the same workspace as twenty thousand.
    constexpr int kAsnormChunkRows = 16384;
    const int chunk = std::min(N, kAsnormChunkRows);
    const size_t tmp_bytes = (size_t)chunk * ld * sizeof(float);
    int rc = ws_ensure(0, tmp_bytes);
    if (rc) return rc;
    static PerDeviceOnce configured;
    if (configured.first()) {
        SKB_CUDA_CHECK(cudaFuncSetAttribute(topk_stats_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    }
    for (int r0 = 0; r0 < N; r0 += chunk) {
        const int rows = std::min(chunk, N - r0);
        rc = score_gemm_general(X_dev + (size_t)r0 * D, cohort_dev, rows, C, D, nullptr, nullptr, 1.f, nullptr, nullptr, 0.f, 1.f, 1.f, 3, 0,
                                g_ws.tmp, ld, tmp_bytes, st);
        if (rc) return rc;
        SKB_CUDA_CHECK(launch_kernel(false, topk_stats_kernel, dim3(rows), dim3(256), C * sizeof(unsigned), st, g_ws.tmp, C, ld, top_k,
                                     mean_dev + r0, std_dev + r0));
    }
    return SKB_OK;
}

int skb_asnorm_apply(const float* X_dev, int N, int D, const float* mean_dev, const float* std_dev, float* out_dev,
                     void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    const size_t tmp_bytes = (size_t)2 * N * sizeof(float);
    int rc = ws_ensure(0, tmp_bytes);
    if (rc) return rc;
    float* ra = g_ws.tmp;
    float* r = ra + N;
    SKB_CUDA_CHECK(launch_kernel(false, asnorm_terms_kernel, dim3((N + 255) / 256), dim3(256), 0, st, mean_dev, std_dev, N, ra, r));
    return score_gemm_general(X_dev, X_dev, N, N, D, ra, ra, 0.f, r, r, 0.f, 1.f, 30.f, 3, 0, out_dev, N, tmp_bytes, st);
}

// Row panel of the as-norm matrix for the multi-GPU path (SURVEY.md 8e): the rows [row0, row0 + n_rows) of
// out[i][j] = 0.5*(S_ij - mean_i)/std_i + 0.5*(S_ij - mean_j)/std_j; the statistics of ALL N embeddings are needed
// (all-gathered by the caller), the embeddings of the panel's rows are Xrows_dev = X_dev + row0 * D.
int skb_asnorm_apply_panel(const float* X_dev, int N, int D, int row0, int n_rows, const float* mean_dev, const float* std_dev,
                           float* out_dev, int64_t ld_out, void* stream) {
    if (!X_dev || !mean_dev || !std_dev || !out_dev || row0 < 0 || n_rows <= 0 || row0 + n_rows > N || ld_out < N) {
        set_last_error(__FILE__, __LINE__, "asnorm_apply_panel: bad arguments");
        return SKB_ERR_ARG;
    }
    cudaStream_t st = (cudaStream_t)stream;
    const size_t tmp_bytes = (size_t)2 * N * sizeof(float);
    int rc = ws_ensure(0, tmp_bytes);
    if (rc) return rc;
    float* ra = g_ws.tmp;
    float* r = ra + N;
    SKB_CUDA_CHECK(launch_kernel(false, asnorm_terms_kernel, dim3((N + 255) / 256), dim3(256), 0, st, mean_dev, std_dev, N, ra, r));
    return score_gemm_general(X_dev + (size_t)row0 * D, X_dev, n_rows, N, D, ra + row0, ra, 0.f, r + row0, r, 0.f, 1.f, 30.f, 3, 0,
                              out_dev, ld_out, tmp_bytes, st);
}

int skb_score_pairs(const float* E_dev, const float* T_dev, int Ne, int Nt, int D, const int32_t* rows_dev, const int32_t* cols_dev,
                    int64_t n_pairs, const float* rowterm_dev, const float* colterm_dev, float cst, float alpha, const float* mean_e_dev,
                    const float* std_e_dev, const float* mean_t_dev, const float* std_t_dev, float* out_dev, void* stream) {
    const int n_stats = (mean_e_dev != nullptr) + (std_e_dev != nullptr) + (mean_t_dev != nullptr) + (std_t_dev != nullptr);
    if (Ne < 0 || Nt < 0 || D < 0 || n_pairs < 0 || (n_stats != 0 && n_stats != 4)) {
        set_last_error(__FILE__, __LINE__, "score_pairs: bad arguments (negative size, or some but not all four as-norm vectors)");
        return SKB_ERR_ARG;
    }
    if (n_pairs == 0) return SKB_OK;
    if (!E_dev || !T_dev || !rows_dev || !cols_dev || !out_dev || D == 0) {
        set_last_error(__FILE__, __LINE__, "score_pairs: null operand or D = 0");
        return SKB_ERR_ARG;
    }
    const long long ctas = (n_pairs + kPairsPerCta - 1) / kPairsPerCta;
    if (ctas > 0x7fffffffLL) {
        set_last_error(__FILE__, __LINE__, "score_pairs: too many trials for one launch");
        return SKB_ERR_ARG;
    }
    const PairArgs a{E_dev, T_dev, Ne, Nt, D, rows_dev, cols_dev, (long long)n_pairs, rowterm_dev, colterm_dev, cst, alpha,
                     mean_e_dev, std_e_dev, mean_t_dev, std_t_dev, out_dev};
    const bool vec = (D & 3) == 0 && (reinterpret_cast<uintptr_t>(E_dev) & 15) == 0 && (reinterpret_cast<uintptr_t>(T_dev) & 15) == 0;
    cudaStream_t st = (cudaStream_t)stream;
    SKB_CUDA_CHECK(launch_kernel(true, vec ? score_pairs_kernel<true> : score_pairs_kernel<false>, dim3((unsigned)ctas), dim3(kPairThreads), 0,
                                 st, a));
    return SKB_OK;
}

}  // extern "C"
