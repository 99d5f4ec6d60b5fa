// FLAC decoding of the feed path (RFC 9639, up to 24 bits per sample): what torchaudio.load / soundfile.read do for the
// reference's .flac inputs (sidekit/nnet/xsets.py:419-464, sidekit/bin/extract_xvectors.py:37-72), for a whole batch of
// files in three launches.  The host parses the metadata blocks only (sidekit_b200/flac.py); frames are found here.
//
//  1. flac_scan_kernel, one thread per input byte.  A byte that starts a sync code and a frame header whose CRC-8 checks is
//     a candidate: its thread parses every subframe of the frame (Rice codes are walked, nothing is predicted), byte-aligns,
//     and checks the CRC-16 over the whole frame.  flen[p] = the frame's byte length when all of this holds, else 0.
//     A sync code plus a valid CRC-8 inside residual data is thereby rejected unless a whole frame parses from it with a
//     valid CRC-16, and even then step 2 only accepts it where the previous frame ends.
//  2. flac_chain_kernel, one thread per file: walks flen from the end of the metadata, each frame starting where the
//     previous one ends, checks the frame / sample numbers and the blocking strategy, and stops when the block sizes reach
//     STREAMINFO's total (trailing bytes, e.g. an ID3v1 tag, are ignored).  It lists the accepted frames (start byte, first
//     sample) and sets the file's status; a broken chain, a wrong number or a wrong total is a corrupt file.
//  3. flac_decode_kernel: one thread per accepted frame decodes the subframes channel 0 needs (channel 1 too for side/right
//     and mid/side) with 64-bit prediction sums, and writes channel 0 as float32 int / 2^(bps - 1) into the packed output.
//
// Every read goes through a reader bounded by the file's byte range (bytes past it read as zero and mark the parse as
// overrun); every write is inside [first sample, first sample + block size) of a frame whose range step 2 checked against
// the file's total.
#include "sidekit_b200.h"
#include "common.cuh"

namespace skb {

// one row of the file table (files_dev), all int64: byte range of the frames in the input buffer, output offset, STREAMINFO
struct FlacFile {
    long long begin, end, out_off, total, slot_base, slot_cap, rate, channels, bps;
};
struct FlacSlot {
    long long pos, first;
};
static_assert(sizeof(FlacFile) == 9 * sizeof(int64_t), "files_dev rows are 9 x int64");

constexpr int kScanThreads = 256;
constexpr int kChainThreads = 64;
constexpr int kDecodeThreads = 128;
// frames per warp in the decode kernel: the work of a frame is one serial walk, so a few frames per warp trade SIMD width
// for more warps to hide the latency of that walk
constexpr int kDecodeLanes = 8;

__constant__ int kRates[12] = {0, 88200, 176400, 192000, 8000, 16000, 22050, 24000, 32000, 44100, 48000, 96000};
__constant__ int kSampleSizes[8] = {0, 8, 12, 0, 16, 20, 24, 0};
__constant__ int kFixedCoefs[5][4] = {{0, 0, 0, 0}, {1, 0, 0, 0}, {2, -1, 0, 0}, {3, -3, 1, 0}, {4, -6, 4, -1}};

struct FrameHdr {
    int bs, rate, assign, nch, bps, variable, len;   // len: header bytes, CRC-8 included
    unsigned long long number;
};

__device__ __forceinline__ unsigned crc8_update(unsigned crc, unsigned byte) {
    crc ^= byte;
#pragma unroll
    for (int k = 0; k < 8; ++k) crc = (crc & 0x80) ? ((crc << 1) ^ 0x07) & 0xFF : (crc << 1) & 0xFF;
    return crc;
}

// Frame header at byte p (RFC 9639 section 9.1), checked against STREAMINFO: false unless every field is valid, the
// CRC-8 checks and bits per sample, channel count and (when coded) sample rate agree with the file.
__device__ bool parse_header(const uint8_t* __restrict__ in, long long p, const FlacFile& F, FrameHdr& h) {
    const long long avail = F.end - p;
    auto rd = [&](int i) -> unsigned { return i < avail ? (unsigned)__ldg(in + p + i) : 0u; };
    if (avail < 6 || rd(0) != 0xFF || (rd(1) & 0xFE) != 0xF8) return false;
    h.variable = rd(1) & 1;
    const unsigned b2 = rd(2), b3 = rd(3);
    const int bs_code = b2 >> 4, rate_code = b2 & 15, assign = b3 >> 4, ss = (b3 >> 1) & 7;
    if (bs_code == 0 || rate_code == 15 || assign > 10 || ss == 3 || ss == 7 || (b3 & 1)) return false;
    // coded number: UTF-8-like, 1-7 bytes (section 9.1.5)
    const unsigned c0 = rd(4);
    int n;
    unsigned long long v;
    if (c0 < 0x80) { n = 1; v = c0; }
    else if ((c0 & 0xE0) == 0xC0) { n = 2; v = c0 & 0x1F; }
    else if ((c0 & 0xF0) == 0xE0) { n = 3; v = c0 & 0x0F; }
    else if ((c0 & 0xF8) == 0xF0) { n = 4; v = c0 & 0x07; }
    else if ((c0 & 0xFC) == 0xF8) { n = 5; v = c0 & 0x03; }
    else if ((c0 & 0xFE) == 0xFC) { n = 6; v = c0 & 0x01; }
    else if (c0 == 0xFE) { n = 7; v = 0; }
    else return false;
    if (!h.variable && n > 6) return false;                  // a frame number has at most 31 bits
    for (int i = 1; i < n; ++i) {
        const unsigned c = rd(4 + i);
        if ((c & 0xC0) != 0x80) return false;
        v = (v << 6) | (c & 0x3F);
    }
    h.number = v;
    int i = 4 + n;
    if (bs_code == 1) h.bs = 192;
    else if (bs_code <= 5) h.bs = 576 << (bs_code - 2);
    else if (bs_code == 6) { h.bs = (int)rd(i) + 1; i += 1; }
    else if (bs_code == 7) { h.bs = (int)((rd(i) << 8) | rd(i + 1)) + 1; i += 2; }
    else h.bs = 256 << (bs_code - 8);
    int rate;
    if (rate_code == 0) rate = (int)F.rate;
    else if (rate_code < 12) rate = kRates[rate_code];
    else if (rate_code == 12) { rate = (int)rd(i) * 1000; i += 1; }
    else if (rate_code == 13) { rate = (int)((rd(i) << 8) | rd(i + 1)); i += 2; }
    else { rate = (int)((rd(i) << 8) | rd(i + 1)) * 10; i += 2; }
    if (i + 1 > avail) return false;
    unsigned crc = 0;
    for (int k = 0; k < i; ++k) crc = crc8_update(crc, rd(k));
    if (crc != rd(i)) return false;
    h.len = i + 1;
    h.bps = ss == 0 ? (int)F.bps : kSampleSizes[ss];
    h.assign = assign;
    h.nch = assign <= 7 ? assign + 1 : 2;
    h.rate = rate;
    return h.bps == F.bps && h.nch == F.channels && rate == F.rate;
}

// MSB-first bit reader over [pos, end): bytes at or past `end` read as zero, and consuming them makes ok() false.
struct BitReader {
    const uint8_t* __restrict__ in;
    long long next, end, left;       // next byte to load, end of the file's range, bits left before the end (< 0: overrun)
    unsigned long long buf;          // nb valid bits, left-aligned
    int nb;
    __device__ BitReader(const uint8_t* in_, long long pos, long long end_)
        : in(in_), next(pos), end(end_), left((end_ - pos) * 8), buf(0), nb(0) {}
    __device__ __forceinline__ void refill() {
        while (nb <= 56) {
            const unsigned long long b = next < end ? (unsigned long long)__ldg(in + next) : 0ull;
            ++next;
            buf |= b << (56 - nb);
            nb += 8;
        }
    }
    __device__ __forceinline__ unsigned get(int n) {            // 0 <= n <= 32
        if (n == 0) return 0u;
        refill();
        const unsigned v = (unsigned)(buf >> (64 - n));
        buf <<= n;
        nb -= n;
        left -= n;
        return v;
    }
    __device__ __forceinline__ int get_signed(int n) {
        if (n == 0) return 0;
        return (int)(get(n) << (32 - n)) >> (32 - n);
    }
    __device__ __forceinline__ unsigned unary() {               // zeros before the next one bit
        unsigned q = 0;
        for (;;) {
            refill();
            if (buf) {
                const int z = __clzll(buf);
                buf = (buf << z) << 1;
                nb -= z + 1;
                left -= z + 1;
                return q + z;
            }
            q += nb;
            left -= nb;
            nb = 0;
            if (left < 0) return q;
        }
    }
    __device__ __forceinline__ bool ok() const { return left >= 0; }
    __device__ __forceinline__ bool align() { return get(nb & 7) == 0u; }    // zero padding to the next byte
    __device__ __forceinline__ long long byte_pos() const { return next - nb / 8; }   // valid when byte-aligned
};

// Where a decoded channel goes.  kStoreInt keeps the int sample in the output word for the partner channel, the other
// modes write channel 0 as float (directly, or rebuilt from the stored word for side/right and mid/side).
enum EmitMode { kNone = 0, kStoreInt, kDirect, kSideRight, kMidSide };
struct Emit {
    float* out;
    float scale;
    int mode, wasted;
};
__device__ __forceinline__ void emit(const Emit& e, int i, int v) {
    v = (int)((unsigned)v << e.wasted);
    switch (e.mode) {
        case kStoreInt: reinterpret_cast<int*>(e.out)[i] = v; break;
        case kDirect: e.out[i] = (float)v * e.scale; break;
        case kSideRight: e.out[i] = (float)(reinterpret_cast<const int*>(e.out)[i] + v) * e.scale; break;
        case kMidSide: {
            const int mid = (int)((unsigned)reinterpret_cast<const int*>(e.out)[i] << 1) | (v & 1);
            e.out[i] = (float)((mid + v) >> 1) * e.scale;
            break;
        }
        default: break;
    }
}

// FIXED / LPC subframe after its header (section 9.2.5, 9.2.6) and its residual (9.2.7).  MAXO = 0: parse only (warm-up,
// coefficients and residual are read and dropped); MAXO > 0: order <= MAXO, history and coefficients live in registers,
// h[0] the newest sample, c[j] multiplies h[j], sums in 64 bits.
template <int MAXO>
__device__ bool predicted(BitReader& br, int bs, int sbps, int order, bool lpc, const Emit& e) {
    constexpr int N = MAXO > 0 ? MAXO : 1;
    int h[N], c[N];
#pragma unroll
    for (int j = 0; j < N; ++j) h[j] = c[j] = 0;
    for (int i = 0; i < order; ++i) {
        const int v = br.get_signed(sbps);
        if (MAXO > 0) {
            emit(e, i, v);
#pragma unroll
            for (int j = N - 1; j > 0; --j) h[j] = h[j - 1];
            h[0] = v;
        }
    }
    int shift = 0;
    if (lpc) {
        const int prec = (int)br.get(4) + 1;
        if (prec == 16) return false;
        shift = br.get_signed(5);
        if (shift < 0) return false;
        if (MAXO > 0) {
#pragma unroll
            for (int j = 0; j < N; ++j) c[j] = j < order ? br.get_signed(prec) : 0;
        } else {
            for (int j = 0; j < order; ++j) br.get_signed(prec);
        }
    } else if (MAXO > 0) {
#pragma unroll
        for (int j = 0; j < N; ++j) c[j] = j < 4 ? kFixedCoefs[order][j] : 0;
    }
    if (!br.ok()) return false;
    // residual
    const int method = (int)br.get(2);
    if (method > 1) return false;
    const int porder = (int)br.get(4);
    const int pbits = method ? 5 : 4, esc = method ? 31 : 15;
    const int psize = bs >> porder;
    if ((psize << porder) != bs || psize < order) return false;
    int i = order;
    for (int part = 0; part < (1 << porder); ++part) {
        const int n = part == 0 ? psize - order : psize;
        const int k = (int)br.get(pbits);
        const int w = k == esc ? (int)br.get(5) : 0;
        for (int t = 0; t < n; ++t, ++i) {
            int r;
            if (k == esc) {
                r = br.get_signed(w);
            } else {
                const unsigned u = (br.unary() << k) | br.get(k);
                r = (int)(u >> 1) ^ -(int)(u & 1);
            }
            if (MAXO > 0) {
                long long sum = 0;
#pragma unroll
                for (int j = 0; j < N; ++j) sum += (long long)c[j] * h[j];
                const int s = r + (int)(sum >> shift);
                emit(e, i, s);
#pragma unroll
                for (int j = N - 1; j > 0; --j) h[j] = h[j - 1];
                h[0] = s;
            }
        }
        if (!br.ok()) return false;
    }
    return true;
}

// One subframe (section 9.2) of sbps bits per sample (the side channel's extra bit included).  kParse: only walk it.
template <bool kParse>
__device__ bool subframe(BitReader& br, int bs, int sbps, Emit e) {
    if (br.get(1)) return false;
    const int type = (int)br.get(6);
    int wasted = 0;
    if (br.get(1)) wasted = (int)br.unary() + 1;
    if (!br.ok() || wasted >= sbps) return false;
    sbps -= wasted;
    e.wasted = wasted;
    if (type == 0) {                                             // CONSTANT
        const int v = br.get_signed(sbps);
        if (!kParse)
            for (int i = 0; i < bs; ++i) emit(e, i, v);
        return br.ok();
    }
    if (type == 1) {                                             // VERBATIM
        for (int i = 0; i < bs; ++i) {
            const int v = br.get_signed(sbps);
            if (!kParse) emit(e, i, v);
        }
        return br.ok();
    }
    int order;
    bool lpc;
    if (type >= 8 && type <= 12) { order = type - 8; lpc = false; }
    else if (type >= 32) { order = type - 31; lpc = true; }
    else return false;
    if (order > bs) return false;
    if (kParse) return predicted<0>(br, bs, sbps, order, lpc, e);
    if (order <= 4) return predicted<4>(br, bs, sbps, order, lpc, e);
    if (order <= 8) return predicted<8>(br, bs, sbps, order, lpc, e);
    if (order <= 16) return predicted<16>(br, bs, sbps, order, lpc, e);
    return predicted<32>(br, bs, sbps, order, lpc, e);
}

__device__ __forceinline__ int side_bit(int assign, int ch) {
    return (assign == 8 && ch == 1) || (assign == 9 && ch == 0) || (assign == 10 && ch == 1);
}

// index of the file whose [key_lo, key_hi) holds x; rows sorted by key
__device__ __forceinline__ int find_file(const FlacFile* __restrict__ files, int n_files, long long x, bool by_slot) {
    int lo = 0, hi = n_files - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        const long long key = by_slot ? files[mid].slot_base : files[mid].begin;
        if (key <= x) lo = mid; else hi = mid - 1;
    }
    return lo;
}

__global__ void __launch_bounds__(kScanThreads) flac_scan_kernel(const uint8_t* __restrict__ in, long long n_bytes,
                                                                 const FlacFile* __restrict__ files, int n_files,
                                                                 int* __restrict__ flen) {
    __shared__ uint16_t crc16_table[256];
    {
        unsigned c = threadIdx.x << 8;
#pragma unroll
        for (int k = 0; k < 8; ++k) c = (c & 0x8000) ? (c << 1) ^ 0x8005 : c << 1;
        crc16_table[threadIdx.x] = (uint16_t)c;
    }
    __syncthreads();
    const long long p = (long long)blockIdx.x * kScanThreads + threadIdx.x;
    if (p >= n_bytes) return;
    int len = 0;
    if (__ldg(in + p) == 0xFF && p + 1 < n_bytes && (__ldg(in + p + 1) & 0xFE) == 0xF8) {
        const FlacFile F = files[find_file(files, n_files, p, false)];
        FrameHdr h;
        if (p < F.end && parse_header(in, p, F, h)) {
            BitReader br(in, p + h.len, F.end);
            bool ok = true;
            for (int ch = 0; ch < h.nch && ok; ++ch) ok = subframe<true>(br, h.bs, h.bps + side_bit(h.assign, ch), Emit{nullptr, 0.f, kNone, 0});
            ok = ok && br.align() && br.ok();
            const long long e = br.byte_pos() + 2;
            if (ok && e <= F.end) {
                unsigned crc = 0;
                for (long long q = p; q < e; ++q) crc = ((crc << 8) ^ crc16_table[((crc >> 8) ^ __ldg(in + q)) & 0xFF]) & 0xFFFF;
                if (crc == 0) len = (int)(e - p);
            }
        }
    }
    flen[p] = len;
}

__global__ void __launch_bounds__(kChainThreads) flac_chain_kernel(const uint8_t* __restrict__ in, const FlacFile* __restrict__ files,
                                                                   int n_files, const int* __restrict__ flen,
                                                                   FlacSlot* __restrict__ slots, int* __restrict__ nframes,
                                                                   int* __restrict__ status) {
    const int f = blockIdx.x * kChainThreads + threadIdx.x;
    if (f >= n_files) return;
    const FlacFile F = files[f];
    long long pos = F.begin, sample = 0;
    int k = 0, st = SKB_FLAC_OK, variable = 0, bs0 = 0, prev_bs = 0;
    while (sample < F.total) {
        FrameHdr h;
        const int len = pos < F.end ? flen[pos] : 0;
        if (len <= 0 || !parse_header(in, pos, F, h)) { st = SKB_FLAC_BAD_FRAME; break; }
        if (k == 0) { variable = h.variable; bs0 = h.bs; }
        // fixed blocking: the frame number counts frames and every frame but the last has the first one's size;
        // variable blocking: the number is the frame's first sample
        const bool number_ok = variable ? h.number == (unsigned long long)sample
                                        : h.number == (unsigned long long)k && (k == 0 || prev_bs == bs0);
        if (h.variable != variable || !number_ok) { st = SKB_FLAC_BAD_NUMBER; break; }
        if (sample + h.bs > F.total) { st = SKB_FLAC_BAD_LENGTH; break; }
        if (k >= F.slot_cap) { st = SKB_FLAC_BAD_LENGTH; break; }
        slots[F.slot_base + k] = FlacSlot{pos, sample};
        sample += h.bs;
        prev_bs = h.bs;
        pos += len;
        ++k;
    }
    nframes[f] = st == SKB_FLAC_OK ? k : 0;
    status[f] = st;
}

__global__ void __launch_bounds__(kDecodeThreads) flac_decode_kernel(const uint8_t* __restrict__ in, const FlacFile* __restrict__ files,
                                                                     int n_files, const FlacSlot* __restrict__ slots,
                                                                     const int* __restrict__ nframes, long long n_slots,
                                                                     float* __restrict__ out) {
    const int lane = threadIdx.x & 31;
    if (lane >= kDecodeLanes) return;
    const long long slot = (((long long)blockIdx.x * kDecodeThreads + threadIdx.x) >> 5) * kDecodeLanes + lane;
    if (slot >= n_slots) return;
    const int f = find_file(files, n_files, slot, true);
    const FlacFile F = files[f];
    if (slot - F.slot_base >= nframes[f]) return;
    const FlacSlot s = slots[slot];
    FrameHdr h;
    if (!parse_header(in, s.pos, F, h) || s.first + h.bs > F.total) return;     // both checked by the chain already
    BitReader br(in, s.pos + h.len, F.end);
    const float scale = 1.0f / (float)(1 << (h.bps - 1));
    float* dst = out + F.out_off + s.first;
    const bool pair = h.assign == 9 || h.assign == 10;
    subframe<false>(br, h.bs, h.bps + side_bit(h.assign, 0), Emit{dst, scale, pair ? kStoreInt : kDirect, 0});
    if (pair) subframe<false>(br, h.bs, h.bps + side_bit(h.assign, 1), Emit{dst, scale, h.assign == 9 ? kSideRight : kMidSide, 0});
}

}  // namespace skb

using namespace skb;

extern "C" int64_t skb_flac_workspace_bytes(int64_t n_bytes, int n_files, int64_t n_slots) {
    if (n_bytes < 0 || n_files < 0 || n_slots < 0) return -1;
    return ((n_bytes * 4 + 15) / 16) * 16 + n_slots * (int64_t)sizeof(FlacSlot) + (int64_t)n_files * 4;
}

extern "C" int skb_flac_decode(const uint8_t* bytes_dev, int64_t n_bytes, const int64_t* files_dev, int n_files, int64_t n_slots,
                               void* work_dev, int64_t work_bytes, float* out_dev, int32_t* status_dev, void* stream) {
    if (!bytes_dev || !files_dev || !work_dev || !out_dev || !status_dev || n_bytes <= 0 || n_files <= 0 || n_slots <= 0 ||
        work_bytes < skb_flac_workspace_bytes(n_bytes, n_files, n_slots) || reinterpret_cast<uintptr_t>(work_dev) % 16) {
        set_last_error(__FILE__, __LINE__, "flac_decode: bad arguments");
        return SKB_ERR_ARG;
    }
    cudaStream_t st = (cudaStream_t)stream;
    const FlacFile* files = reinterpret_cast<const FlacFile*>(files_dev);
    int* flen = reinterpret_cast<int*>(work_dev);
    FlacSlot* slots = reinterpret_cast<FlacSlot*>(reinterpret_cast<uint8_t*>(work_dev) + ((n_bytes * 4 + 15) / 16) * 16);
    int* nframes = reinterpret_cast<int*>(slots + n_slots);
    SKB_CUDA_CHECK(launch_kernel(false, flac_scan_kernel, dim3((unsigned)((n_bytes + kScanThreads - 1) / kScanThreads)),
                                 kScanThreads, 0, st, bytes_dev, (long long)n_bytes, files, n_files, flen));
    SKB_CUDA_CHECK(launch_kernel(false, flac_chain_kernel, dim3((unsigned)((n_files + kChainThreads - 1) / kChainThreads)),
                                 kChainThreads, 0, st, bytes_dev, files, n_files, (const int*)flen, slots, nframes, status_dev));
    const long long warps = (n_slots + kDecodeLanes - 1) / kDecodeLanes;
    const long long per_block = kDecodeThreads / 32;
    SKB_CUDA_CHECK(launch_kernel(false, flac_decode_kernel, dim3((unsigned)((warps + per_block - 1) / per_block)), kDecodeThreads, 0,
                                 st, bytes_dev, files, n_files, (const FlacSlot*)slots, (const int*)nframes, (long long)n_slots,
                                 out_dev));
    return SKB_OK;
}
