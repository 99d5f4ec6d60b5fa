// Sample-rate conversion of the feed path: torchaudio.transforms.Resample(orig_freq, new_freq) as the reference calls it
// on every file whose rate differs from the model's (sidekit/nnet/xsets.py:435, :452; sidekit/bin/extract_xvectors.py:144).
//
// Algorithm (torchaudio.functional._get_sinc_resample_kernel / _apply_sinc_resample_kernel): with the rates divided by
// their gcd (orig, new), output sample j = q * new + ph is the FIR
//     y[j] = sum_k bank[ph][k] * x[q * orig + k - width],      k in [0, 2 * width + orig),  x = 0 outside [0, L)
// where bank[ph] is a Hann-windowed sinc sampled at the ph-th fractional delay.  Only ~2 * width of the 2 * width + orig
// taps of a phase lie inside the window (the others are clamped to its edge, where cos^2(pi / 2) ~ 4e-33), so the host
// hands the kernel a COMPACT bank: per phase its first in-window tap and `ntap` consecutive coefficients (zero padded).
// 44.1 kHz -> 16 kHz: 36 multiply-adds per output instead of 475.
//
// The kernel is HBM-bound in principle (4 B read per input sample, 4 B written per output sample, each once); in practice
// the shared-memory pipe sets its speed (one 128-byte wavefront per clock and SM: every multiply-add needs one input
// sample from shared memory), so the layout is chosen to spend exactly one conflict-free wavefront per 32 multiply-adds
// on the samples and a quarter of one on the coefficients:
//  * a CTA produces `pcta` whole periods (pcta * new_r consecutive outputs) of one waveform from an input window staged
//    in shared memory with coalesced loads; the bank stays in shared memory tap-major ([tap][phase]);
//  * a work item is (phase ph, period qb) and the lanes of a warp walk consecutive PERIODS of one phase: the coefficient
//    is a broadcast and the samples are orig_r words apart (conflict-free for odd orig_r -- 441, 147, 3, 1 ...);
//  * each thread computes kResBlock outputs of its phase (periods qb, qb + Qb, ...) per coefficient load;
//  * results go through a padded shared tile ([period][new_r + 1]) and leave the CTA as fully coalesced stores (for
//    new_r <= 2 the lanes' outputs are adjacent already and are stored directly).
#include "sidekit_b200.h"
#include "common.cuh"

#include <stdlib.h>

namespace skb {

constexpr int kOutPerCta = 2048;       // target outputs per CTA (rounded down to whole periods); sweep in profiles/r01g_resample.txt
constexpr int kResThreads = 256;
constexpr int kResBlock = 4;           // outputs per thread and coefficient load

struct ResampleWave {
    long long in_off, in_len, out_off, out_len;
};

// dynamic shared memory: bank_t [ntap][new_r] | start [new_r] (int) | window [win_len] | tile [pcta][new_r + 1]
__global__ void __launch_bounds__(kResThreads) resample_kernel(const float* __restrict__ in, float* __restrict__ out,
                                                               const ResampleWave* __restrict__ waves, int orig_r, int new_r,
                                                               int width, int ntap, const float* __restrict__ bank,
                                                               const int* __restrict__ start, int pcta, int win_len) {
    extern __shared__ __align__(16) uint8_t smem_raw[];
    float* bank_t = reinterpret_cast<float*>(smem_raw);
    int* start_s = reinterpret_cast<int*>(bank_t + (size_t)ntap * new_r);
    float* win = reinterpret_cast<float*>(start_s + new_r);
    float* tile = win + win_len;
    const ResampleWave w = waves[blockIdx.y];
    const long long q0 = (long long)blockIdx.x * pcta;
    const long long j0 = q0 * new_r;
    if (j0 >= w.out_len) return;
    for (int i = threadIdx.x; i < ntap * new_r; i += kResThreads) bank_t[i] = __ldg(bank + i);     // [tap][phase]
    for (int i = threadIdx.x; i < new_r; i += kResThreads) start_s[i] = start[i];
    // input window of this run: samples [x0, x0 + win_len) of the zero-extended waveform
    const long long x0 = q0 * orig_r - width;
    const float* src = in + w.in_off;
    for (int i = threadIdx.x; i < win_len; i += kResThreads) {
        const long long s = x0 + i;
        win[i] = (s >= 0 && s < w.in_len) ? __ldg(src + s) : 0.f;
    }
    __syncthreads();
    const int Qb = (pcta + kResBlock - 1) / kResBlock;
    const int tstride = new_r + 1;
    const bool use_tile = new_r > 2;
    float* dst = out + w.out_off + j0;
    for (int idx = threadIdx.x; idx < new_r * Qb; idx += kResThreads) {
        const int ph = idx / Qb, qb = idx - ph * Qb;
        const float* bp = bank_t + ph;
        const float* xp[kResBlock];
        float acc[kResBlock];
#pragma unroll
        for (int r = 0; r < kResBlock; ++r) {
            const int q = min(qb + r * Qb, pcta - 1);            // surplus slots recompute the last period (never stored)
            xp[r] = win + q * orig_r + start_s[ph];
            acc[r] = 0.f;
        }
        for (int k = 0; k < ntap; ++k) {
            const float c = bp[k * new_r];
#pragma unroll
            for (int r = 0; r < kResBlock; ++r) acc[r] = fmaf(c, xp[r][k], acc[r]);
        }
#pragma unroll
        for (int r = 0; r < kResBlock; ++r) {
            const int q = qb + r * Qb;
            if (q >= pcta) continue;
            if (use_tile) tile[q * tstride + ph] = acc[r];
            else if ((long long)q * new_r + ph < w.out_len - j0) dst[q * new_r + ph] = acc[r];      // new_r <= 2: coalesced as is
        }
    }
    if (!use_tile) return;
    __syncthreads();
    const int n_out = (int)min((long long)pcta * new_r, w.out_len - j0);
    for (int o = threadIdx.x; o < n_out; o += kResThreads) {
        const int q = o / new_r;
        dst[o] = tile[q * tstride + (o - q * new_r)];
    }
}
}  // namespace skb

using namespace skb;

extern "C" int skb_resample(const float* in_dev, const int64_t* wave_meta_dev, int n_wav, int64_t max_out, int orig_r, int new_r,
                            int width, const float* bank_dev, const int32_t* start_dev, int ntap, float* out_dev, void* stream) {
    if (!in_dev || !out_dev || !wave_meta_dev || !bank_dev || !start_dev || n_wav <= 0 || n_wav > 65535 || max_out < 0 ||
        orig_r <= 0 || new_r <= 0 || width <= 0 || ntap <= 0 || ntap > 2 * width + orig_r) {
        set_last_error(__FILE__, __LINE__, "resample: bad arguments");
        return SKB_ERR_ARG;
    }
    if (max_out == 0) return SKB_OK;
    cudaStream_t st = (cudaStream_t)stream;
    // a CTA takes pcta whole periods; its taps span pcta * orig_r + 2 * width input samples
    const int pcta = kOutPerCta / new_r > 0 ? kOutPerCta / new_r : 1;
    const long long win_len = (long long)pcta * orig_r + 2 * width;
    const size_t smem = ((size_t)ntap * new_r + new_r + (size_t)win_len + (new_r > 2 ? (size_t)pcta * (new_r + 1) : 0)) * 4;
    if (smem > 200 * 1024) {
        set_last_error(__FILE__, __LINE__, "resample: rate ratio too irregular for the shared-memory bank (reduce the rates by their gcd)");
        return SKB_ERR_ARG;
    }
    static_assert(sizeof(ResampleWave) == 4 * sizeof(int64_t), "wave_meta_dev rows are 4 x int64");
    SKB_CUDA_CHECK(cudaFuncSetAttribute(resample_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const long long per_cta = (long long)pcta * new_r;
    dim3 grid((unsigned)((max_out + per_cta - 1) / per_cta), (unsigned)n_wav);
    SKB_CUDA_CHECK(launch_kernel(false, resample_kernel, grid, kResThreads, smem, st, in_dev, out_dev,
                                 reinterpret_cast<const ResampleWave*>(wave_meta_dev), orig_r, new_r, width, ntap, bank_dev, start_dev, pcta,
                                 (int)win_len));
    return SKB_OK;
}
