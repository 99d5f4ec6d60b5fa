// Uncompressed audio of the feed path (WAV and NIST SPHERE, every PCM encoding): what torchaudio.load / soundfile.read do
// for the reference's .wav / .sph inputs (sidekit/nnet/xsets.py:419-464, sidekit/bin/extract_xvectors.py:37-72), for a
// whole batch of files in one launch.  The host parses the containers (sidekit_b200/pcm.py) and stages every file's
// sample bytes; this kernel converts channel 0 of each to float32 in the packed output.
//
// Work unit: a tile of kPcmTile consecutive frames of one file, one warp per tile.  Tiles are numbered file after file
// (the table's first-tile column, a prefix sum the host computes); a warp finds its file by binary search.  Stores are
// coalesced: lane l writes frames l, l + 32, ... of the tile.  Mono 16-bit little-endian data whose bytes start 16-byte
// aligned (the host aligns every file's data) is read with one 16-byte load per lane for every whole tile and passed to
// the coalesced store through shared memory; everything else is read byte by byte, bounded by the file's frame count.
#include "sidekit_b200.h"
#include "common.cuh"

namespace skb {

// one row of the file table (files_dev), all int64
struct PcmFile {
    long long offset, frames, channels, encoding, bytes, big_endian, out_off, first_tile;
};
static_assert(sizeof(PcmFile) == 8 * sizeof(int64_t), "files_dev rows are 8 x int64");

constexpr int kPcmTile = 256;                    // frames per tile = 32 lanes x 8
constexpr int kPcmThreads = 256;                 // 8 warps, 8 tiles per block

// G.711 expansion to the 16-bit value, as the Sun g711.c routines (and libsndfile's / audioop's tables) compute it
__device__ __forceinline__ int ulaw_to_s16(unsigned u) {
    u = ~u & 0xFF;
    int t = ((u & 0x0F) << 3) + 0x84;
    t <<= (u & 0x70) >> 4;
    return (u & 0x80) ? 0x84 - t : t - 0x84;
}
__device__ __forceinline__ int alaw_to_s16(unsigned a) {
    a ^= 0x55;
    int t = (a & 0x0F) << 4;
    const int seg = (a & 0x70) >> 4;
    if (seg == 0) t += 8;
    else t = (t + 0x108) << (seg - 1);
    return (a & 0x80) ? t : -t;
}

__device__ __forceinline__ float sample_at(const uint8_t* __restrict__ p, const PcmFile& F) {
    const int nb = (int)F.bytes;
    unsigned long long v = 0;
    for (int i = 0; i < nb; ++i) {
        const unsigned long long b = __ldg(p + i);
        v |= b << (8 * (F.big_endian ? nb - 1 - i : i));
    }
    switch ((int)F.encoding) {
    case SKB_PCM_INT: {                          // signed, nb = 1..4: x / 2^(8 nb - 1)
        const int sh = 64 - 8 * nb;
        const long long x = (long long)(v << sh) >> sh;
        return __int2float_rn((int)x) * __int_as_float((127 - (8 * nb - 1)) << 23);
    }
    case SKB_PCM_U8:
        return (float)((int)v - 128) * (1.0f / 128.0f);
    case SKB_PCM_FLOAT:
        return nb == 8 ? __double2float_rn(__longlong_as_double((long long)v)) : __uint_as_float((unsigned)v);
    case SKB_PCM_ULAW:
        return (float)ulaw_to_s16((unsigned)v) * (1.0f / 32768.0f);
    default:
        return (float)alaw_to_s16((unsigned)v) * (1.0f / 32768.0f);
    }
}

__global__ void __launch_bounds__(kPcmThreads) pcm_decode_kernel(const uint8_t* __restrict__ in, const PcmFile* __restrict__ files,
                                                                 int n_files, long long n_tiles, float* __restrict__ out) {
    __shared__ __align__(16) float stage[kPcmThreads / 32][kPcmTile];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const long long tile = (long long)blockIdx.x * (kPcmThreads / 32) + warp;
    if (tile >= n_tiles) return;
    int lo = 0, hi = n_files - 1;                // last file whose first tile <= tile (0-frame files own no tile)
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (files[mid].first_tile <= tile) lo = mid;
        else hi = mid - 1;
    }
    const PcmFile F = files[lo];
    const long long f0 = (tile - F.first_tile) * kPcmTile;
    const long long n = min((long long)kPcmTile, F.frames - f0);
    float* dst = out + F.out_off + f0;
    const bool vec = F.channels == 1 && F.bytes == 2 && F.encoding == SKB_PCM_INT && !F.big_endian &&
                     reinterpret_cast<uintptr_t>(in + F.offset) % 16 == 0;
    if (vec && n == kPcmTile) {
        const uint4 w = __ldg(reinterpret_cast<const uint4*>(in + F.offset + f0 * 2) + lane);
        const unsigned u[4] = {w.x, w.y, w.z, w.w};
        float v[8];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            v[2 * k] = (float)(short)(u[k] & 0xFFFF) * (1.0f / 32768.0f);
            v[2 * k + 1] = (float)(short)(u[k] >> 16) * (1.0f / 32768.0f);
        }
        float4* s = reinterpret_cast<float4*>(&stage[warp][lane * 8]);
        s[0] = make_float4(v[0], v[1], v[2], v[3]);
        s[1] = make_float4(v[4], v[5], v[6], v[7]);
        __syncwarp();
#pragma unroll
        for (int j = 0; j < kPcmTile / 32; ++j) dst[lane + 32 * j] = stage[warp][lane + 32 * j];
        return;
    }
    const long long stride = F.channels * F.bytes;
    for (int j = lane; j < n; j += 32) dst[j] = sample_at(in + F.offset + (f0 + j) * stride, F);
}

}  // namespace skb

using namespace skb;

extern "C" int skb_pcm_decode(const uint8_t* bytes_dev, const int64_t* files_dev, int n_files, int64_t n_tiles, float* out_dev,
                              void* stream) {
    if (!files_dev || n_files <= 0 || n_tiles < 0 || (n_tiles > 0 && (!bytes_dev || !out_dev))) {   // no tile: no sample to read or write
        set_last_error(__FILE__, __LINE__, "pcm_decode: bad arguments");
        return SKB_ERR_ARG;
    }
    constexpr long long per_block = kPcmThreads / 32;
    const unsigned blocks = (unsigned)(n_tiles > 0 ? (n_tiles + per_block - 1) / per_block : 1);
    SKB_CUDA_CHECK(launch_kernel(false, pcm_decode_kernel, dim3(blocks), kPcmThreads, 0, (cudaStream_t)stream, bytes_dev,
                                 reinterpret_cast<const PcmFile*>(files_dev), n_files, (long long)n_tiles, out_dev));
    return SKB_OK;
}
