// Shared device helpers for the sm_100a kernels: mbarrier, 1-D bulk async copy (TMA engine,
// SASS UBLKCP), tcgen05 (alloc / mma / commit / ld) and UMMA descriptor construction.
// Everything is inline PTX; no CUTLASS/CuTe dependency.
#pragma once
#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>
#include <atomic>

namespace skb {

constexpr int kNumSMs = 148;

// Per-device one-time configuration (cudaFuncSetAttribute is per device / context) and per-device workspaces:
// a process may use several GPUs one after the other (cosine_scoring(device=...), Xtractor.to("cuda:1")).
constexpr int kMaxDevices = 64;
inline int current_device() {
    int d = 0;
    if (cudaGetDevice(&d) != cudaSuccess || d < 0 || d >= kMaxDevices) d = 0;
    return d;
}
struct PerDeviceOnce {
    bool done[kMaxDevices] = {};
    bool first() {                       // true exactly once per device (a benign race repeats an idempotent call)
        const int d = current_device();
        if (done[d]) return false;
        done[d] = true;
        return true;
    }
};

#define SKB_CUDA_CHECK(expr)                                                                  \
    do {                                                                                      \
        cudaError_t _e = (expr);                                                              \
        if (_e != cudaSuccess) {                                                              \
            skb::set_last_error(__FILE__, __LINE__, cudaGetErrorString(_e));                  \
            return SKB_ERR_CUDA;                                                              \
        }                                                                                     \
    } while (0)

void set_last_error(const char* file, int line, const char* msg);

// ----------------------------------------------------------------------------- programmatic dependent launch (PDL)
// The kernels of the per-block chain (conv1 -> channel sums -> border sums -> SE partial means -> SE FC -> conv2) depend on
// each other one after the other.  Launched with the programmatic-stream-serialization attribute, kernel k+1 is scheduled
// as soon as the CTAs of kernel k have exited (without waiting for the end-of-grid flush), its CTAs run their prologue
// (barrier init, TMEM allocation, constant weights), and pdl_wait() -- executed by every such kernel before it reads or
// writes anything another kernel touches -- blocks until kernel k has completed and its writes are visible.
// Measured (profiles/r01g_pdl.txt): 8.53 -> 8.45 ms per HalfResNet34 step, e2e +1.5 %.  An EARLY trigger
// (griddepcontrol.launch_dependents at the top of every kernel) lets the whole chain park on the SMs while conv1 still runs
// and is slower (8.7-8.8 ms), so the implicit trigger at CTA exit is what the chain uses.
// SKB_NO_PDL=1 launches everything with plain stream order (A/B knob); pdl_wait() is then a no-op.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
// explicit trigger: the next kernel of the stream may be scheduled once every CTA of this grid has got here -- used by
// se_border_kernel AFTER its own pdl_wait, so that the channel-total pass that follows (which needs nothing from the border
// sums) runs beside it instead of behind it
__device__ __forceinline__ void pdl_trigger_now() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
bool pdl_enabled();

// ----------------------------------------------------------------------------- kernel launch
// Every kernel of the library is launched here, so that skb_kernel_launches() counts each one and SKB_SYNC_CHECK=1
// synchronises the stream after each one: an execution fault is then reported at the SKB_CUDA_CHECK of the launch that
// caused it (compute-sanitizer is not always available).  pdl = true launches with the programmatic-stream-serialization
// attribute (see above; SKB_NO_PDL=1 turns it off), pdl = false in plain stream order.
extern std::atomic<long long> g_launches;
bool sync_check_enabled();
template <typename... KArgs, typename... Args>
inline cudaError_t launch_kernel(bool pdl, void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st,
                                 Args&&... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    if (pdl) {
        attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[0].val.programmaticStreamSerializationAllowed = pdl_enabled() ? 1 : 0;
        cfg.attrs = attr;
        cfg.numAttrs = 1;
    }
    const cudaError_t e = cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
    if (e != cudaSuccess) return e;
    ++g_launches;
    return sync_check_enabled() ? cudaStreamSynchronize(st) : cudaSuccess;
}

// ----------------------------------------------------------------------------- shared-memory address
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

// ----------------------------------------------------------------------------- mbarrier
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_barrier_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
// Bounded wait: a protocol bug must surface as a trap (launch error), never as a hung GPU.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    if (mbar_try_wait(bar, parity)) return;
    const long long t0 = clock64();
    while (!mbar_try_wait(bar, parity)) {
        if (clock64() - t0 > 4000000000LL) {   // ~2 s at 1.9 GHz
            printf("skb: mbarrier timeout block (%d,%d) thread %d parity %u\n", blockIdx.x, blockIdx.y,
                   threadIdx.x, parity);
            __trap();
        }
    }
}

// ----------------------------------------------------------------------------- bulk async copy (global -> shared)
__device__ __forceinline__ void bulk_g2s(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(smem_dst)),
                 "l"(gsrc), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

// ----------------------------------------------------------------------------- tcgen05
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

template <int kCols>
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_result) {   // whole warp
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_result)),
                 "n"(kCols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
template <int kCols>
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr) {        // whole warp (the allocating one)
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(kCols) : "memory");
}

// One elected lane of a fully converged warp (deterministic: the same lane every time for the same mask).
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "elect.sync _|p, 0xffffffff;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(pred));
    return pred != 0;
}

// Shared-memory matrix descriptor, K-major, no swizzle ("interleaved" canonical layout):
//   core matrix = 8 rows x 16 bytes stored as 128 contiguous bytes,
//   LBO = byte distance between the two 16-byte K halves of one K=16 instruction,
//   SBO = byte distance between consecutive 8-row groups along M/N.
// Bits: [0,14) start>>4, [16,30) LBO>>4, [32,46) SBO>>4, [46,48) version=1 (sm_100), [61,64) layout=0.
__device__ __forceinline__ uint64_t umma_desc_kmajor_noswz(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    uint64_t d = 0;
    d |= static_cast<uint64_t>((smem_addr >> 4) & 0x3FFF);
    d |= static_cast<uint64_t>((lbo_bytes >> 4) & 0x3FFF) << 16;
    d |= static_cast<uint64_t>((sbo_bytes >> 4) & 0x3FFF) << 32;
    d |= static_cast<uint64_t>(1) << 46;
    return d;
}

// Instruction descriptor for kind::f16: fp32 accumulate, A/B both K-major, 16-bit inputs.
//   bits [4,6) c_format (1 = f32), [7,10) a_format, [10,13) b_format (0 = f16, 1 = bf16),
//   [17,23) N>>3, [24,29) M>>4.
__host__ __device__ constexpr uint32_t umma_idesc_f16(int M, int N, bool bf16) {
    return (1u << 4) | ((bf16 ? 1u : 0u) << 7) | ((bf16 ? 1u : 0u) << 10) | (static_cast<uint32_t>(N >> 3) << 17) |
           (static_cast<uint32_t>(M >> 4) << 24);
}

__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                         uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// A operand in TENSOR MEMORY (lane = row, 8 columns per K = 16 slab of 16-bit elements), B from shared memory: the MMA then
// reads only B through the shared-memory pipe.
__device__ __forceinline__ void umma_f16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}" ::"r"(tmem_d),
        "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// shared memory -> tensor memory: 128 rows x 32 bytes (one K = 16 slab in the canonical K-major layout the MMA descriptors
// use) into 128 lanes x 8 columns.  Executes in issue order with the tcgen05.mma of the same thread.
__device__ __forceinline__ void tmem_cp_128x256b(uint32_t taddr, uint64_t sdesc) {
    asm volatile("tcgen05.cp.cta_group::1.128x256b [%0], %1;" ::"r"(taddr), "l"(sdesc) : "memory");
}
// Arrive on an mbarrier once every tcgen05 op previously issued by this thread has completed.
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
                 : "memory");
}

// TMEM -> registers: this warp's 32 lanes x 32 consecutive fp32 columns (thread = one accumulator row).
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float (&v)[32]) {
    uint32_t r[32];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
          "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
          "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr)
        : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}

// Same, 16 consecutive fp32 columns.
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float (&v)[16]) {
    uint32_t r[16];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr)
        : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}

// ----------------------------------------------------------------------------- 16-bit packing
// fp16 range guard (SURVEY.md 7 "Precision"): the fp16 conversion SATURATES (F2FP.SATFINITE, same cost as the plain
// convert) instead of producing +-inf, and the kernels that store activations keep a running max |x| of what they stored
// (one HMNMX2 per two values); a thread that saw a saturated value bumps a device counter at its exit, which the host
// surfaces as an error (skb_xtractor_overflow_count).  bf16 has the fp32 exponent range and needs neither.
template <bool kBf16>
__device__ __forceinline__ uint32_t pack2(float lo, float hi) {
    if (kBf16) {
        __nv_bfloat162 t = __floats2bfloat162_rn(lo, hi);
        return *reinterpret_cast<uint32_t*>(&t);
    } else {
        uint32_t r;
        asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
        return r;
    }
}
__device__ __forceinline__ void track16(uint32_t packed, uint32_t& running_max) {      // fp16 pairs only
    const __half2 m = __hmax2(__habs2(*reinterpret_cast<const __half2*>(&packed)), *reinterpret_cast<const __half2*>(&running_max));
    running_max = *reinterpret_cast<const uint32_t*>(&m);
}
__device__ __forceinline__ void track16(const uint4& o, uint32_t& running_max) {
    track16(o.x, running_max); track16(o.y, running_max); track16(o.z, running_max); track16(o.w, running_max);
}
__device__ __forceinline__ bool saturated16(uint32_t running_max) {                     // 0x7BFF = 65504, the largest finite fp16
    return (running_max & 0x7fffu) >= 0x7bffu || ((running_max >> 16) & 0x7fffu) >= 0x7bffu;
}
template <bool kBf16>
__device__ __forceinline__ float2 unpack2(uint32_t u) {
    if (kBf16) {
        return __bfloat1622float2(*reinterpret_cast<__nv_bfloat162*>(&u));
    } else {
        return __half22float2(*reinterpret_cast<__half2*>(&u));
    }
}

__device__ __forceinline__ long long shfl_xor_ll(long long v, int off) {
    const int lo = __shfl_xor_sync(0xffffffffu, (int)(v & 0xffffffffll), off);
    const int hi = __shfl_xor_sync(0xffffffffu, (int)(v >> 32), off);
    return ((long long)hi << 32) | (unsigned int)lo;
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

}  // namespace skb
