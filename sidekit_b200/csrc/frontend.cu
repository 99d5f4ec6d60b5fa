// Fused front-end: pre-emphasis -> framing (reflect pad, periodic Hann) -> real FFT in shared
// memory -> power -> sparse triangular Mel filterbank -> log(. + 1e-6) [-> DCT for MFCC], then a
// per-(utterance, coefficient) CMVN pass.  One kernel replaces PreEmphasis conv1d + torch.stft (cuFFT)
// + |.|^2 + mel matmul + log of sidekit/nnet/preprocessor.py:267-285 (log-Mel) and :113-124 (MFCC);
// the 513 x T spectrogram never touches HBM.
//
// FFT: a real frame of n_fft samples is packed as n_fft/2 complex points z[n] = f[2n] + i f[2n+1],
// transformed by a radix-8 decimation-in-frequency FFT (digit-reversed output), and unpacked with
//   X[k] = (Z[k] + conj Z[N/2-k])/2 - (i/2) e^{-2 pi i k/n_fft} (Z[k] - conj Z[N/2-k]).
// The window sits at the start of the frame instead of the centre: a circular shift only changes
// the phase, and only |X|^2 is used.
#include "sidekit_b200.h"
#include "common.cuh"
#include "layers.cuh"

namespace skb {

struct FrontendParams {
    const float* wave;        // concatenated utterances
    const long long* wave_off;// [B] start of each utterance in `wave`
    const int* wave_len;      // [B] samples
    const long long* feat_off;// [B] start (in frames) of each utterance in the frame-major output
    const int* n_frames;      // [B]
    float* out;               // [sum T][n_out] frame-major
    const float* window;      // [win]
    const float2* tw_half;    // [NC] e^{-2 pi i m / NC}, NC = n_fft/2
    const float2* tw_full;    // [NC+1] e^{-2 pi i k / n_fft}
    const int* mel_lo;        // [n_mels] first FFT bin of each filter
    const int* mel_cnt;       // [n_mels] number of bins
    const int* mel_ofs;       // [n_mels] offset into mel_w
    const float* mel_w;       // filter weights, concatenated
    const float* dct;         // [n_mels][n_out] or nullptr (log-Mel)
    int n_mels, n_out;
    int hop, win;
    int n_w;                  // number of (concatenated) mel filter weights
    int dct_smem_off;         // offset (in floats, multiple of 4) of the DCT matrix inside the kernel's shared memory
    float preemph;
};

__device__ __forceinline__ float2 cmul(float2 a, float2 b) { return make_float2(a.x * b.x - a.y * b.y, a.x * b.y + a.y * b.x); }
__device__ __forceinline__ float2 cadd(float2 a, float2 b) { return make_float2(a.x + b.x, a.y + b.y); }
__device__ __forceinline__ float2 csub(float2 a, float2 b) { return make_float2(a.x - b.x, a.y - b.y); }
__device__ __forceinline__ float2 cmul_mi(float2 a) { return make_float2(a.y, -a.x); }   // a * (-i)

// ---- register-resident FFT of N = 16 / 32 points (radix-2 DIF, fully unrolled; output in bit-reversed order) ------------
// cos / sin of 2 pi j / 32, j = 0 .. 15 (w_32^j = cos - i sin); w_16^j = w_32^{2j}
__device__ constexpr float kCos32[16] = {1.f, 0.98078528040323044913f, 0.92387953251128675613f, 0.83146961230254523708f,
                                         0.70710678118654752440f, 0.55557023301960222474f, 0.38268343236508977173f,
                                         0.19509032201612826785f, 0.f, -0.19509032201612826785f, -0.38268343236508977173f,
                                         -0.55557023301960222474f, -0.70710678118654752440f, -0.83146961230254523708f,
                                         -0.92387953251128675613f, -0.98078528040323044913f};
__device__ constexpr float kSin32[16] = {0.f, 0.19509032201612826785f, 0.38268343236508977173f, 0.55557023301960222474f,
                                         0.70710678118654752440f, 0.83146961230254523708f, 0.92387953251128675613f,
                                         0.98078528040323044913f, 1.f, 0.98078528040323044913f, 0.92387953251128675613f,
                                         0.83146961230254523708f, 0.70710678118654752440f, 0.55557023301960222474f,
                                         0.38268343236508977173f, 0.19509032201612826785f};

template <int N>
__host__ __device__ constexpr int brev(int i) {      // bit reversal over log2(N) bits
    int r = 0;
    for (int b = 1; b < N; b <<= 1) { r = (r << 1) | (i & 1); i >>= 1; }
    return r;
}

template <int N>
__device__ __forceinline__ void fft_dif(float2 (&a)[N]) {
#pragma unroll
    for (int half = N / 2; half >= 1; half >>= 1) {
#pragma unroll
        for (int blk = 0; blk < N; blk += 2 * half) {
#pragma unroll
            for (int j = 0; j < half; ++j) {
                const float2 u = a[blk + j], v = a[blk + j + half];
                a[blk + j] = cadd(u, v);
                const float2 d = csub(u, v);
                const int t = j * (16 / half);           // twiddle w_{2 half}^j = w_32^t
                if (t == 0) a[blk + j + half] = d;
                else if (t == 8) a[blk + j + half] = cmul_mi(d);
                else a[blk + j + half] = cmul(d, make_float2(kCos32[t], -kSin32[t]));
            }
        }
    }
}

// NC complex points per frame, one WARP per frame, NC = A x 32 with A = NC / 32 (16 or 32), four-step FFT:
//   1. lane n2 takes the A points z[n1 * 32 + n2] STRAIGHT FROM THE WAVEFORM (pre-emphasis, reflect padding and window
//      applied on the fly: no staging pass) and transforms them in registers (fft_dif<A>);
//   2. multiplies by the twiddles w_NC^{n2 k1} (a [k1][n2] table in shared memory: conflict-free) and writes
//      S[k1][n2] (row stride 33: conflict-free both ways);
//   3. lane k1 < A reads its row, transforms the 32 points in registers (fft_dif<32>) and stores Z[k1 + A k2] in natural order.
// Two trips through shared memory instead of the five of the radix-8 in-place version; the passes are separated by
// __syncwarp only, so the WPC warps of a CTA never wait for each other.
template <int NC, int WPC>
__global__ void __launch_bounds__(WPC * 32, (640 / (WPC * 32)) > 0 ? 640 / (WPC * 32) : 1) frontend_kernel(const FrontendParams p, int frames_per_cta) {
    constexpr int A = NC / 32;
    // Frames per warp and trip.  With A = 16 (log-Mel, n_fft 1024) the 32-point transforms of step 3 occupy only 16 lanes:
    // the warp takes TWO frames per trip and runs both frames' step 3 together (lanes 0-15 / 16-31), which halves the
    // issue slots of the heaviest step (the kernel is issue-bound, profiles/r01f_ncu_frontend_logmel.txt).
    constexpr int FPW = A == 16 ? 2 : 1;
    constexpr int ZS = (A * 33 > NC + 2 ? A * 33 : NC + 2);      // complex slots per frame buffer: S[A][33] or Z[NC] / pwr[NC + 1]
    // Every table a frame touches lives in shared memory (twiddles, window, sparse mel filterbank, DCT): read through
    // L1 / L2 they were 52 KB per frame on the MFCC front-end, 2.8 GB of L2 reads for 0.38 GB of audio
    // (profiles/r01c_ncu_frontend_mfcc_before.txt).
    extern __shared__ __align__(16) uint8_t fsm[];
    float2* tw = reinterpret_cast<float2*>(fsm);                 // [A][32]: w_NC^{n2 k1}
    float2* twf = tw + NC;                                       // [NC + 1] (+1 pad): e^{-2 pi i k / n_fft}
    float2* zall = twf + NC + 2;                                 // [WPC][FPW][ZS]
    float* melall = reinterpret_cast<float*>(zall + WPC * FPW * ZS);   // [WPC][n_mels]
    float* s_win = melall + WPC * p.n_mels;                      // [win]
    float* s_melw = s_win + p.win;                               // [n_w]
    int* s_lo = reinterpret_cast<int*>(s_melw + p.n_w);          // [n_mels] x 3: first bin, count, weight offset
    int* s_cnt = s_lo + p.n_mels;
    int* s_ofs = s_cnt + p.n_mels;
    float* s_dct = reinterpret_cast<float*>(fsm) + p.dct_smem_off;   // [n_mels][n_out], 16-byte aligned, or unused
    const int b = blockIdx.y;
    const int T = p.n_frames[b];
    const int t_begin = blockIdx.x * frames_per_cta;
    if (t_begin >= T) return;
    const int t_end = min(T, t_begin + frames_per_cta);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (int i = threadIdx.x; i < NC; i += blockDim.x) tw[i] = p.tw_half[((i >> 5) * (i & 31)) & (NC - 1)];   // k1 = i / 32, n2 = i % 32
    for (int i = threadIdx.x; i <= NC; i += blockDim.x) twf[i] = p.tw_full[i];
    for (int i = threadIdx.x; i < p.win; i += blockDim.x) s_win[i] = p.window[i];
    for (int i = threadIdx.x; i < p.n_w; i += blockDim.x) s_melw[i] = p.mel_w[i];
    for (int i = threadIdx.x; i < p.n_mels; i += blockDim.x) { s_lo[i] = p.mel_lo[i]; s_cnt[i] = p.mel_cnt[i]; s_ofs[i] = p.mel_ofs[i]; }
    if (p.dct != nullptr)
        for (int i = threadIdx.x; i < p.n_mels * p.n_out; i += blockDim.x) s_dct[i] = p.dct[i];
    __syncthreads();
    const float* x = p.wave + p.wave_off[b];
    const int L = p.wave_len[b];
    float2* zwarp = zall + warp * FPW * ZS;
    float* mel = melall + warp * p.n_mels;
    const int half_win = p.win >> 1;

    for (int frame0 = t_begin + warp * FPW; frame0 < t_end; frame0 += WPC * FPW) {
      // ---- steps 0-2 for each frame of the trip (frame validity is warp-uniform)
#pragma unroll
      for (int f = 0; f < FPW; ++f) {
        const int frame = frame0 + f;
        if (frame >= t_end) break;
        float2* z = zwarp + f * ZS;
        // ---- step 0: the frame's samples (pre-emphasis, reflect padding, window) into the frame buffer.  All the loads
        // of the loop are independent, so eight of them are in flight per lane; fetched inside step 1 the compiler
        // serialised them behind the FFT's registers (one L2 / HBM round trip per pair of points: 32 % of the MFCC
        // kernel's stall samples, profiles/r01d_ncu_frontend_mfcc.txt).
        float* ybuf = reinterpret_cast<float*>(z);
        {
            const int i_base = p.hop * frame - half_win;
#pragma unroll 8
            for (int n = lane; n < p.win; n += 32) {
                int i = i_base + n;
                if (i < 0) i = -i;
                if (i >= L) i = 2 * (L - 1) - i;
                const float cur = __ldg(x + i);
                const float prev = __ldg(x + (i == 0 ? 1 : i - 1));
                ybuf[n] = (cur - p.preemph * prev) * s_win[n];
            }
        }
        __syncwarp();
        // ---- step 1: A points per lane (sample pairs 2 (n1 * 32 + lane), +1), transformed in registers
        {
            float2 a[A];
#pragma unroll
            for (int n1 = 0; n1 < A; ++n1) {
                // win <= n_fft / 2 (checked by frontend_launch): the upper half of the points is the zero padding, a
                // compile-time fact that removes the first butterfly stage
                const int n = 2 * (n1 * 32 + lane);
                float2 v = make_float2(0.f, 0.f);
                if (n1 < A / 2) {
                    if (n + 1 < p.win) v = *reinterpret_cast<const float2*>(ybuf + n);
                    else if (n < p.win) v.x = ybuf[n];
                }
                a[n1] = v;
            }
            __syncwarp();                                        // step 2 overwrites the buffer
            fft_dif<A>(a);
            // ---- step 2: twiddle and transpose through shared memory
#pragma unroll
            for (int r = 0; r < A; ++r) {
                const int k1 = brev<A>(r);                       // a[r] = Y[k1]
                float2 y = a[r];
                if (k1 != 0) y = cmul(y, tw[k1 * 32 + lane]);
                z[k1 * 33 + lane] = y;
            }
        }
      }
        __syncwarp();
        // ---- step 3: 32 points per lane, natural-order store.  A = 32: lane k1 of the single frame; A = 16: lanes 0-15 take
        // the rows of the trip's first frame, lanes 16-31 those of the second
        {
            float2 c[32];
            const int f3 = FPW == 2 ? (lane >> 4) : 0, k1 = FPW == 2 ? (lane & 15) : lane;
            const bool act = k1 < A && frame0 + f3 < t_end;
            float2* z3 = zwarp + f3 * ZS;
            if (act) {
#pragma unroll
                for (int n2 = 0; n2 < 32; ++n2) c[n2] = z3[k1 * 33 + n2];
            }
            __syncwarp();                                        // every row is in registers before Z overwrites S
            if (act) {
                fft_dif<32>(c);
#pragma unroll
                for (int r = 0; r < 32; ++r) z3[k1 + A * brev<32>(r)] = c[r];     // Z[k1 + A k2]
            }
        }
        __syncwarp();
      // ---- power spectrum, mel, log (and DCT) per frame of the trip
#pragma unroll
      for (int f = 0; f < FPW; ++f) {
        const int frame = frame0 + f;
        if (frame >= t_end) break;
        float2* z = zwarp + f * ZS;
        // unpack the real spectrum, take |X|^2 for k = 0..NC and store it in natural order into a power buffer that
        // aliases z (all reads first).  Bins k and NC - k share everything but two signs:
        //   X[k]      = ((s.x + wd.y) - i (wd.x - s.y)) / 2,   X[NC - k] = conj-symmetric with wd -> conj(wd),
        //   s = Z[k] + conj Z[NC-k],  wd = e^{-2 pi i k / n_fft} (Z[k] - conj Z[NC-k]),
        // so one pass over k = 0 .. NC/2 yields both halves (k = 0 gives the DC and the Nyquist bin).
        constexpr int kHalfIt = NC / 64;            // k = lane + 32 c < NC / 2
        float pw_lo[kHalfIt], pw_hi[kHalfIt], pw_mid = 0.f;
#pragma unroll
        for (int c = 0; c < kHalfIt; ++c) {
            const int k = lane + c * 32;
            const float2 zk = z[k];
            const float2 zr = z[(NC - k) & (NC - 1)];
            const float2 zc = make_float2(zr.x, -zr.y);
            const float2 s = cadd(zk, zc), d = csub(zk, zc);
            const float2 wd = cmul(twf[k], d);
            const float re = 0.5f * (s.x + wd.y), im = 0.5f * (s.y - wd.x);
            const float re2 = 0.5f * (s.x - wd.y), im2 = 0.5f * (s.y + wd.x);
            pw_lo[c] = re * re + im * im;
            pw_hi[c] = re2 * re2 + im2 * im2;
        }
        if (lane == 0) {                            // k = NC / 2 is its own mirror image
            const float2 zk = z[NC / 2];
            const float2 zc = make_float2(zk.x, -zk.y);
            const float2 s = cadd(zk, zc), d = csub(zk, zc);
            const float2 wd = cmul(twf[NC / 2], d);
            const float re = 0.5f * (s.x + wd.y), im = 0.5f * (s.y - wd.x);
            pw_mid = re * re + im * im;
        }
        __syncwarp();
        float* pwr = reinterpret_cast<float*>(z);
#pragma unroll
        for (int c = 0; c < kHalfIt; ++c) {
            const int k = lane + c * 32;
            pwr[k] = pw_lo[c];
            pwr[NC - k] = pw_hi[c];
        }
        if (lane == 0) pwr[NC / 2] = pw_mid;
        __syncwarp();
        float* dst = p.out + (size_t)(p.feat_off[b] + frame) * p.n_out;
        // sparse mel filterbank: lane = mel bin for the full rounds of 32; the remaining n_mels % 32 bins -- the widest
        // filters (40 FFT bins each on the MFCC front-end, where only 4 lanes had work) -- are split over several lanes
        // each and combined with a fixed-order shuffle tree
        const int full = p.n_mels & ~31;
        for (int m = lane; m < full; m += 32) {
            const int lo = s_lo[m], c = s_cnt[m];
            const float* w = s_melw + s_ofs[m];
            float acc = 0.f;
            for (int i = 0; i < c; ++i) acc = fmaf(pwr[lo + i], w[i], acc);
            const float lm = logf(acc + 1e-6f);
            if (p.dct == nullptr) dst[m] = lm;
            else mel[m] = lm;
        }
        const int rest = p.n_mels - full;
        if (rest > 0) {
            int P = 1;
            while (P < rest) P <<= 1;
            const int lanes_per = 32 / P;                       // 8 for 100 mels, 2 for 80
            const int mi = lane / lanes_per, part = lane - mi * lanes_per;
            const int m = full + mi;
            float acc = 0.f;
            if (mi < rest) {
                const int lo = s_lo[m], c = s_cnt[m];
                const float* w = s_melw + s_ofs[m];
                const int chunk = (c + lanes_per - 1) / lanes_per;
                const int i1 = min(c, (part + 1) * chunk);
                for (int i = part * chunk; i < i1; ++i) acc = fmaf(pwr[lo + i], w[i], acc);
            }
            for (int off = lanes_per >> 1; off >= 1; off >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, off);
            if (mi < rest && part == 0) {
                const float lm = logf(acc + 1e-6f);
                if (p.dct == nullptr) dst[m] = lm;
                else mel[m] = lm;
            }
        }
        if (p.dct != nullptr) {
            __syncwarp();
            // lane l computes the four consecutive outputs 4l .. 4l+3: one 16-byte load of a DCT row per mel bin (rows are
            // 16-byte aligned when n_out is a multiple of 4), the log-Mel value broadcast from shared memory
            if ((p.n_out & 3) == 0) {
                const int c4 = lane * 4;
                if (c4 < p.n_out) {
                    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
                    for (int m = 0; m < p.n_mels; ++m) {
                        const float lm = mel[m];
                        const float4 d = *reinterpret_cast<const float4*>(s_dct + (size_t)m * p.n_out + c4);
                        acc.x = fmaf(lm, d.x, acc.x); acc.y = fmaf(lm, d.y, acc.y);
                        acc.z = fmaf(lm, d.z, acc.z); acc.w = fmaf(lm, d.w, acc.w);
                    }
                    *reinterpret_cast<float4*>(dst + c4) = acc;
                }
                if (p.n_out > 128) {      // (never: frontend_launch rejects it)
                }
            } else {
                for (int c = lane; c < p.n_out; c += 32) {
                    float acc = 0.f;
                    for (int m = 0; m < p.n_mels; ++m) acc = fmaf(mel[m], s_dct[m * p.n_out + c], acc);
                    dst[c] = acc;
                }
            }
        }
        __syncwarp();     // the next frame's fill overwrites z / pwr / mel
      }
    }
}

// CMVN (torch.nn.InstanceNorm1d, biased variance, eps 1e-5) statistics per (utterance, coefficient) over time on the
// frame-major buffer: fixed 64-frame chunks summed in double (sum, sum of squares), then combined in chunk order --
// deterministic and, in double, as exact as the two-pass formula.  The normalisation itself is applied by the consumer
// (stem kernel) or by cmvn_apply_kernel.
constexpr int kCmvnChunk = 64;
__global__ void __launch_bounds__(128) cmvn_partial_kernel(const float* __restrict__ feats, const long long* __restrict__ feat_off,
                                                           const int* __restrict__ n_frames, int n_out, int max_chunks,
                                                           double2* __restrict__ part) {
    const int b = blockIdx.y, ch = blockIdx.x, c = threadIdx.x;
    const int T = n_frames[b], t0 = ch * kCmvnChunk;
    if (t0 >= T || c >= n_out) return;
    const int t1 = min(T, t0 + kCmvnChunk);
    const float* f = feats + (size_t)feat_off[b] * n_out + c;
    double s = 0.0, ss = 0.0;
    for (int t = t0; t < t1; ++t) {
        const double v = (double)f[(size_t)t * n_out];
        s += v;
        ss = fma(v, v, ss);
    }
    part[((size_t)b * max_chunks + ch) * n_out + c] = make_double2(s, ss);
}

__global__ void __launch_bounds__(128) cmvn_final_kernel(const double2* __restrict__ part, const int* __restrict__ n_frames, int n_out,
                                                         int max_chunks, float2* __restrict__ cmvn) {
    const int b = blockIdx.x, c = threadIdx.x;
    if (c >= n_out) return;
    const int T = n_frames[b], nch = (T + kCmvnChunk - 1) / kCmvnChunk;
    double s = 0.0, ss = 0.0;
    for (int ch = 0; ch < nch; ++ch) {
        const double2 v = part[((size_t)b * max_chunks + ch) * n_out + c];
        s += v.x;
        ss += v.y;
    }
    const double mean = s / T;
    const double var = fmax(ss / T - mean * mean, 0.0);
    cmvn[(size_t)b * n_out + c] = make_float2((float)mean, (float)(1.0 / sqrt(var + 1e-5)));
}

// in-place normalisation (+ optionally the (B, n_out, t_max) tensor the reference's front-end returns)
__global__ void cmvn_apply_kernel(float* __restrict__ feats, const long long* __restrict__ feat_off, const int* __restrict__ n_frames,
                                  int n_out, const float2* __restrict__ cmvn, float* __restrict__ api_out, int t_max) {
    const int b = blockIdx.y;
    const int T = n_frames[b];
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (long long)T * n_out) return;
    const int t = (int)(idx / n_out), c = (int)(idx - (long long)t * n_out);
    const float2 ms = cmvn[(size_t)b * n_out + c];
    float* f = feats + (size_t)feat_off[b] * n_out;
    const float v = (f[idx] - ms.x) * ms.y;
    f[idx] = v;
    if (api_out) api_out[((size_t)b * n_out + c) * t_max + t] = v;
}

}  // namespace skb

#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <vector>

namespace skb {

int frontend_consts_create(FrontendConsts* fc, int n_fft, int win, int hop, int n_mels, int n_out, const float* window,
                           const float* fb /* [n_fft/2+1][n_mels] */, const float* dct /* [n_mels][n_out] or null */) {
    fc->n_fft = n_fft; fc->win = win; fc->hop = hop; fc->n_mels = n_mels; fc->n_out = n_out;
    const int NC = n_fft / 2, NB = NC + 1;
    std::vector<float2> th(NC), tf(NB);
    for (int i = 0; i < NC; ++i) {
        const double a = -2.0 * M_PI * i / NC;
        th[i] = make_float2((float)cos(a), (float)sin(a));
    }
    for (int k = 0; k < NB; ++k) {
        const double a = -2.0 * M_PI * k / n_fft;
        tf[k] = make_float2((float)cos(a), (float)sin(a));
    }
    std::vector<int> lo(n_mels), cnt(n_mels), ofs(n_mels);
    std::vector<float> w;
    for (int m = 0; m < n_mels; ++m) {
        int first = -1, last = -1;
        for (int k = 0; k < NB; ++k)
            if (fb[(size_t)k * n_mels + m] != 0.f) { if (first < 0) first = k; last = k; }
        lo[m] = first < 0 ? 0 : first;
        cnt[m] = first < 0 ? 0 : last - first + 1;
        ofs[m] = (int)w.size();
        for (int k = 0; k < cnt[m]; ++k) w.push_back(fb[(size_t)(lo[m] + k) * n_mels + m]);
    }
    if (w.empty()) w.push_back(0.f);
    fc->n_w = (int)w.size();
    SKB_CUDA_CHECK(cudaMalloc(&fc->window, win * sizeof(float)));
    SKB_CUDA_CHECK(cudaMemcpy(fc->window, window, win * sizeof(float), cudaMemcpyHostToDevice));
    SKB_CUDA_CHECK(cudaMalloc(&fc->tw_half, NC * sizeof(float2)));
    SKB_CUDA_CHECK(cudaMemcpy(fc->tw_half, th.data(), NC * sizeof(float2), cudaMemcpyHostToDevice));
    SKB_CUDA_CHECK(cudaMalloc(&fc->tw_full, NB * sizeof(float2)));
    SKB_CUDA_CHECK(cudaMemcpy(fc->tw_full, tf.data(), NB * sizeof(float2), cudaMemcpyHostToDevice));
    SKB_CUDA_CHECK(cudaMalloc(&fc->mel_lo, n_mels * sizeof(int)));
    SKB_CUDA_CHECK(cudaMemcpy(fc->mel_lo, lo.data(), n_mels * sizeof(int), cudaMemcpyHostToDevice));
    SKB_CUDA_CHECK(cudaMalloc(&fc->mel_cnt, n_mels * sizeof(int)));
    SKB_CUDA_CHECK(cudaMemcpy(fc->mel_cnt, cnt.data(), n_mels * sizeof(int), cudaMemcpyHostToDevice));
    SKB_CUDA_CHECK(cudaMalloc(&fc->mel_ofs, n_mels * sizeof(int)));
    SKB_CUDA_CHECK(cudaMemcpy(fc->mel_ofs, ofs.data(), n_mels * sizeof(int), cudaMemcpyHostToDevice));
    SKB_CUDA_CHECK(cudaMalloc(&fc->mel_w, w.size() * sizeof(float)));
    SKB_CUDA_CHECK(cudaMemcpy(fc->mel_w, w.data(), w.size() * sizeof(float), cudaMemcpyHostToDevice));
    if (dct) {
        SKB_CUDA_CHECK(cudaMalloc(&fc->dct, (size_t)n_mels * n_out * sizeof(float)));
        SKB_CUDA_CHECK(cudaMemcpy(fc->dct, dct, (size_t)n_mels * n_out * sizeof(float), cudaMemcpyHostToDevice));
    }
    return SKB_OK;
}

void frontend_consts_destroy(FrontendConsts* fc) {
    cudaFree(fc->window); cudaFree(fc->tw_half); cudaFree(fc->tw_full); cudaFree(fc->mel_lo);
    cudaFree(fc->mel_cnt); cudaFree(fc->mel_ofs); cudaFree(fc->mel_w); cudaFree(fc->dct);
    *fc = FrontendConsts();
}

size_t frontend_cmvn_scratch_bytes(const FrontendConsts& fc, int B, int t_max) {
    const int max_chunks = (t_max + kCmvnChunk - 1) / kCmvnChunk;
    return (size_t)B * max_chunks * fc.n_out * sizeof(double2);
}

// feats: frame-major [sum T][n_out]; api_out optional (B, n_out, t_max).
constexpr int kFramesPerWarp = 8;   // frames each warp of a CTA transforms

int frontend_launch(const FrontendConsts& fc, const float* wave, const long long* wave_off, const int* wave_len,
                    const long long* feat_off, const int* n_frames, int B, int t_max, float* feats, float2* cmvn,
                    void* cmvn_part, bool normalise, float* api_out, cudaStream_t stream) {
    FrontendParams p;
    p.wave = wave; p.wave_off = wave_off; p.wave_len = wave_len; p.feat_off = feat_off; p.n_frames = n_frames;
    p.out = feats; p.window = fc.window; p.tw_half = fc.tw_half; p.tw_full = fc.tw_full;
    p.mel_lo = fc.mel_lo; p.mel_cnt = fc.mel_cnt; p.mel_ofs = fc.mel_ofs; p.mel_w = fc.mel_w; p.dct = fc.dct;
    p.n_mels = fc.n_mels; p.n_out = fc.n_out; p.hop = fc.hop; p.win = fc.win; p.preemph = fc.preemph;
    if (fc.n_out > 128) {
        set_last_error(__FILE__, __LINE__, "front-end: more than 128 output coefficients");
        return SKB_ERR_ARG;
    }
    p.n_w = fc.n_w;
    if (fc.win > fc.n_fft / 2) {
        set_last_error(__FILE__, __LINE__, "front-end: the window must not exceed n_fft / 2");
        return SKB_ERR_ARG;
    }
    auto smem_bytes = [&](int NC, int WPC, int* dct_off) {
        const size_t zs = std::max<size_t>((size_t)(NC / 32) * 33, (size_t)NC + 2);      // complex slots per frame buffer (kernel: ZS)
        const size_t fpw = NC / 32 == 16 ? 2 : 1;                                        // frame buffers per warp (kernel: FPW)
        size_t floats = 2 * (size_t)NC + 2 * ((size_t)NC + 2) + 2 * (size_t)WPC * fpw * zs + (size_t)WPC * fc.n_mels + fc.win + fc.n_w +
                        3 * (size_t)fc.n_mels;
        floats = (floats + 3) / 4 * 4;
        *dct_off = (int)floats;
        if (fc.dct) floats += (size_t)fc.n_mels * fc.n_out;
        return floats * sizeof(float);
    };
    if (fc.n_fft == 1024) {
        constexpr int NC = 512, WPC = 8;
        const int frames_per_cta = kFramesPerWarp * WPC;
        dim3 grid((t_max + frames_per_cta - 1) / frames_per_cta, B);
        const size_t smem = smem_bytes(NC, WPC, &p.dct_smem_off);
        static PerDeviceOnce configured;
        if (configured.first()) {
            SKB_CUDA_CHECK(cudaFuncSetAttribute(frontend_kernel<NC, WPC>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
        }
        if (smem > 227 * 1024) {
            set_last_error(__FILE__, __LINE__, "front-end: tables do not fit in shared memory");
            return SKB_ERR_ARG;
        }
        SKB_CUDA_CHECK(launch_kernel(false, frontend_kernel<NC, WPC>, grid, WPC * 32, smem, stream, p, frames_per_cta));
    } else if (fc.n_fft == 2048) {
        // a frame needs 9.3 KB of shared memory and the tables 52 KB: 16 frame-warps in one CTA per SM
        constexpr int NC = 1024, WPC = 16;
        const int frames_per_cta = kFramesPerWarp * WPC;
        dim3 grid((t_max + frames_per_cta - 1) / frames_per_cta, B);
        const size_t smem = smem_bytes(NC, WPC, &p.dct_smem_off);
        static PerDeviceOnce configured;
        if (configured.first()) {
            SKB_CUDA_CHECK(cudaFuncSetAttribute(frontend_kernel<NC, WPC>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
        }
        if (smem > 227 * 1024) {
            set_last_error(__FILE__, __LINE__, "front-end: tables do not fit in shared memory");
            return SKB_ERR_ARG;
        }
        SKB_CUDA_CHECK(launch_kernel(false, frontend_kernel<NC, WPC>, grid, WPC * 32, smem, stream, p, frames_per_cta));
    } else {
        set_last_error(__FILE__, __LINE__, "unsupported n_fft (1024 or 2048)");
        return SKB_ERR_ARG;
    }
    const int max_chunks = (t_max + kCmvnChunk - 1) / kCmvnChunk;
    SKB_CUDA_CHECK(launch_kernel(false, cmvn_partial_kernel, dim3(max_chunks, B), 128, 0, stream, feats, feat_off, n_frames, fc.n_out, max_chunks,
                                 (double2*)cmvn_part));
    SKB_CUDA_CHECK(launch_kernel(false, cmvn_final_kernel, B, 128, 0, stream, (const double2*)cmvn_part, n_frames, fc.n_out, max_chunks, cmvn));
    if (normalise) {
        const long long per_utt = (long long)t_max * fc.n_out;
        SKB_CUDA_CHECK(launch_kernel(false, cmvn_apply_kernel, dim3((unsigned)((per_utt + 255) / 256), B), 256, 0, stream, feats, feat_off, n_frames,
                                     fc.n_out, cmvn, api_out, t_max));
    }
    return SKB_OK;
}

}  // namespace skb
