// cast_kernels.cu -- the I/O casts of the attention path as HBM-bound sm_100a kernels.
//
// Replaces cvt_d2f_avx512 (attention-mpi.c:31-64, fp64->fp32 round-to-nearest-even)
// and cvt_f2d_avx512 (attention-mpi.c:68-101, exact widening); adds the fp64->bf16
// cast that feeds the tensor-core kernel.  Algorithmic traffic: 12 B/element for
// d2f and f2d, 10 B/element for d2bf16.  Each thread moves 16-byte vectors with
// several independent loads in flight; a scalar kernel covers unaligned pointers and tails.
#include <cstring>
#include "common.cuh"
#include "umma_ptx.cuh"

namespace sdpa {

namespace {

constexpr int kCastThreads = 256;

__device__ __forceinline__ double2 ld_stream_f64x2(const double2* p)
{
    double2 v;
    asm volatile("ld.global.nc.L1::no_allocate.v2.f64 {%0, %1}, [%2];" : "=d"(v.x), "=d"(v.y) : "l"(p));
    return v;
}

__device__ __forceinline__ float4 ld_stream_f32x4(const float4* p)
{
    float4 v;
    asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0, %1, %2, %3}, [%4];"
                 : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
                 : "l"(p));
    return v;
}

// Every warp-level load/store below is contiguous across the warp (16 B per lane on the
// wide side), and each thread keeps kUnroll independent loads in flight per step.
constexpr int kUnroll = 4;

// unit = 2 elements: one 16 B fp64 load -> one 8 B fp32 store.
__global__ void __launch_bounds__(kCastThreads)
cvt_d2f_vec_kernel(float2* __restrict__ dst, const double2* __restrict__ src, size_t units)
{
    const size_t total = (size_t)gridDim.x * blockDim.x;
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    for (; i + (kUnroll - 1) * total < units; i += kUnroll * total) {
        double2 v[kUnroll];
#pragma unroll
        for (int u = 0; u < kUnroll; ++u) v[u] = ld_stream_f64x2(src + i + u * total);
#pragma unroll
        for (int u = 0; u < kUnroll; ++u)
            dst[i + u * total] = make_float2(__double2float_rn(v[u].x), __double2float_rn(v[u].y));
    }
    for (; i < units; i += total) {
        const double2 v = ld_stream_f64x2(src + i);
        dst[i] = make_float2(__double2float_rn(v.x), __double2float_rn(v.y));
    }
}

__global__ void __launch_bounds__(kCastThreads)
cvt_d2f_scalar_kernel(float* __restrict__ dst, const double* __restrict__ src, size_t begin, size_t count)
{
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t i = begin + (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += stride)
        dst[i] = __double2float_rn(src[i]);
}

// unit = 4 elements: one 16 B fp32 load -> two 16 B fp64 stores.
__global__ void __launch_bounds__(kCastThreads)
cvt_f2d_vec_kernel(double2* __restrict__ dst, const float4* __restrict__ src, size_t units)
{
    const size_t total = (size_t)gridDim.x * blockDim.x;
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    for (; i + (kUnroll - 1) * total < units; i += kUnroll * total) {
        float4 v[kUnroll];
#pragma unroll
        for (int u = 0; u < kUnroll; ++u) v[u] = ld_stream_f32x4(src + i + u * total);
#pragma unroll
        for (int u = 0; u < kUnroll; ++u) {
            dst[2 * (i + u * total) + 0] = make_double2((double)v[u].x, (double)v[u].y);
            dst[2 * (i + u * total) + 1] = make_double2((double)v[u].z, (double)v[u].w);
        }
    }
    for (; i < units; i += total) {
        const float4 v = ld_stream_f32x4(src + i);
        dst[2 * i + 0] = make_double2((double)v.x, (double)v.y);
        dst[2 * i + 1] = make_double2((double)v.z, (double)v.w);
    }
}

__global__ void __launch_bounds__(kCastThreads)
cvt_f2d_scalar_kernel(double* __restrict__ dst, const float* __restrict__ src, size_t begin, size_t count)
{
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t i = begin + (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += stride)
        dst[i] = (double)src[i];
}

__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi)
{
    // cvt.rn.bf16x2.f32 d, a, b : a -> upper half, b -> lower half
    uint32_t r;
    asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
    return r;
}

// unit = 2 elements: one 16 B fp64 load -> one 4 B bf16x2 store (fp64 -> fp32 RN -> bf16 RN).
__global__ void __launch_bounds__(kCastThreads)
cvt_d2bf16_vec_kernel(uint32_t* __restrict__ dst, const double2* __restrict__ src, size_t units)
{
    const size_t total = (size_t)gridDim.x * blockDim.x;
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    for (; i + (kUnroll - 1) * total < units; i += kUnroll * total) {
        double2 v[kUnroll];
#pragma unroll
        for (int u = 0; u < kUnroll; ++u) v[u] = ld_stream_f64x2(src + i + u * total);
#pragma unroll
        for (int u = 0; u < kUnroll; ++u)
            dst[i + u * total] = pack_bf16x2(__double2float_rn(v[u].x), __double2float_rn(v[u].y));
    }
    for (; i < units; i += total) {
        const double2 v = ld_stream_f64x2(src + i);
        dst[i] = pack_bf16x2(__double2float_rn(v.x), __double2float_rn(v.y));
    }
}

__global__ void __launch_bounds__(kCastThreads)
cvt_d2bf16_scalar_kernel(__nv_bfloat16* __restrict__ dst, const double* __restrict__ src, size_t begin,
                         size_t count)
{
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t i = begin + (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += stride)
        dst[i] = __float2bfloat16_rn(__double2float_rn(src[i]));
}

// fp32 pair -> (hi, lo) bf16 pairs of the split precision: hi = bf16(x32), lo = bf16(x32 - hi): hi + lo carries 16 mantissa
// bits of x32.  For a bf16 x32, hi = x32 and lo = 0.
__device__ __forceinline__ void split_bf16x2(float a, float b, uint32_t& hi, uint32_t& lo)
{
    hi = pack_bf16x2(a, b);
    lo = pack_bf16x2(a - __uint_as_float(hi << 16), b - __uint_as_float(hi & 0xffff0000u));
}
// fp64 -> (hi, lo): x32 = fp32(x) (the reference's own cvt_d2f, mpi.c:31-64) first.  12 B per element like d2f (8 read, 2 + 2 written).
__device__ __forceinline__ void split_bf16x2(double2 v, uint32_t& hi, uint32_t& lo)
{
    split_bf16x2(__double2float_rn(v.x), __double2float_rn(v.y), hi, lo);
}

__global__ void __launch_bounds__(kCastThreads)
cvt_d2bf16x2_vec_kernel(uint32_t* __restrict__ dst_hi, uint32_t* __restrict__ dst_lo, const double2* __restrict__ src, size_t units)
{
    const size_t total = (size_t)gridDim.x * blockDim.x;
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    for (; i + (kUnroll - 1) * total < units; i += kUnroll * total) {
        double2 v[kUnroll];
#pragma unroll
        for (int u = 0; u < kUnroll; ++u) v[u] = ld_stream_f64x2(src + i + u * total);
#pragma unroll
        for (int u = 0; u < kUnroll; ++u) {
            uint32_t hi, lo;
            split_bf16x2(v[u], hi, lo);
            dst_hi[i + u * total] = hi;
            dst_lo[i + u * total] = lo;
        }
    }
    for (; i < units; i += total) {
        uint32_t hi, lo;
        split_bf16x2(ld_stream_f64x2(src + i), hi, lo);
        dst_hi[i] = hi;
        dst_lo[i] = lo;
    }
}

__global__ void __launch_bounds__(kCastThreads)
cvt_d2bf16x2_scalar_kernel(__nv_bfloat16* __restrict__ dst_hi, __nv_bfloat16* __restrict__ dst_lo, const double* __restrict__ src,
                           size_t begin, size_t count)
{
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t i = begin + (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += stride) {
        const float a = __double2float_rn(src[i]);
        const __nv_bfloat16 h = __float2bfloat16_rn(a);
        dst_hi[i] = h;
        dst_lo[i] = __float2bfloat16_rn(a - __bfloat162float(h));
    }
}

// Source element types of the batched cast: fp64 (the reference's operands) and, for typed device passes, fp32 and bf16.
// Unit = 2 elements, loaded as one vector and widened to an fp32 pair (fp64 rounds to nearest even, like cvt_d2f; fp32 and
// bf16 are exact).
template <typename SRC> struct SrcPair;
template <> struct SrcPair<double> {
    using Unit = double2;
    static __device__ __forceinline__ Unit load(const Unit* p) { return ld_stream_f64x2(p); }
    static __device__ __forceinline__ float2 f32(Unit v) { return make_float2(__double2float_rn(v.x), __double2float_rn(v.y)); }
};
template <> struct SrcPair<float> {
    using Unit = float2;
    static __device__ __forceinline__ Unit load(const Unit* p)
    {
        float2 v;
        asm volatile("ld.global.nc.L1::no_allocate.v2.f32 {%0, %1}, [%2];" : "=f"(v.x), "=f"(v.y) : "l"(p));
        return v;
    }
    static __device__ __forceinline__ float2 f32(Unit v) { return v; }
};
template <> struct SrcPair<__nv_bfloat16> {
    using Unit = uint32_t;   // two bf16, the first in the low half
    static __device__ __forceinline__ Unit load(const Unit* p)
    {
        uint32_t v;
        asm volatile("ld.global.nc.L1::no_allocate.b32 %0, [%1];" : "=r"(v) : "l"(p));
        return v;
    }
    static __device__ __forceinline__ float2 f32(Unit v) { return make_float2(__uint_as_float(v << 16), __uint_as_float(v & 0xffff0000u)); }
};

// Several casts into compute precision in ONE launch (the K shard, the V shard and the first Q batch of a device-resident
// call): the segments form one virtual array of 2-element units, so the grid-stride loop has a single tail instead of one
// per operand and two launch gaps disappear from the step.
// MODE 0: fp32, 1: bf16, 2: bf16 hi/lo split (lo array cb.lo_off[seg] 2-element units behind the hi array).  Every mode
// goes through the fp32 pair of SrcPair<SRC>, so an fp32 source gives the bits an fp64 source of the same fp32 values gives.
template <typename SRC, int MODE>
__global__ void __launch_bounds__(kCastThreads) cvt_in_batch_kernel(CastBatch cb)
{
    using P = SrcPair<SRC>;
    using Unit = typename P::Unit;
    const size_t u0 = cb.units[0], u01 = u0 + cb.units[1], all = u01 + cb.units[2];
    const size_t total = (size_t)gridDim.x * blockDim.x;
    auto locate = [&](size_t g, const Unit*& src, void*& dst, size_t& off, size_t& lo) {
        const int seg = g < u0 ? 0 : (g < u01 ? 1 : 2);
        off = g - (seg == 0 ? 0 : (seg == 1 ? u0 : u01));
        src = reinterpret_cast<const Unit*>(cb.src[seg]);
        dst = cb.dst[seg];
        lo = cb.lo_off[seg];
    };
    auto store = [&](void* dst, size_t off, size_t lo, Unit u) {
        const float2 v = P::f32(u);
        if (MODE == 2) {
            uint32_t h, l;
            split_bf16x2(v.x, v.y, h, l);
            reinterpret_cast<uint32_t*>(dst)[off] = h;
            reinterpret_cast<uint32_t*>(dst)[off + lo] = l;
        } else if (MODE == 1) {
            reinterpret_cast<uint32_t*>(dst)[off] = pack_bf16x2(v.x, v.y);
        } else {
            reinterpret_cast<float2*>(dst)[off] = v;
        }
    };
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    for (; i + (kUnroll - 1) * total < all; i += kUnroll * total) {
        Unit v[kUnroll];
        void* d[kUnroll];
        size_t off[kUnroll], lo[kUnroll];
#pragma unroll
        for (int u = 0; u < kUnroll; ++u) {
            const Unit* src;
            locate(i + u * total, src, d[u], off[u], lo[u]);
            v[u] = P::load(src + off[u]);
        }
#pragma unroll
        for (int u = 0; u < kUnroll; ++u) store(d[u], off[u], lo[u], v[u]);
    }
    for (; i < all; i += total) {
        const Unit* src;
        void* d;
        size_t off, lo;
        locate(i, src, d, off, lo);
        store(d, off, lo, P::load(src + off));
    }
}

// Scalar form of one fp32 / bf16 segment (unaligned pointers, odd counts): the same conversions, one element per thread.
template <typename SRC, int MODE>
__global__ void __launch_bounds__(kCastThreads)
cvt_typed_scalar_kernel(void* __restrict__ dst, size_t lo_off, const SRC* __restrict__ src, size_t count)
{
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += stride) {
        const float a = (float)src[i];
        if (MODE == 0) {
            reinterpret_cast<float*>(dst)[i] = a;
        } else {
            __nv_bfloat16* d = reinterpret_cast<__nv_bfloat16*>(dst);
            const __nv_bfloat16 h = __float2bfloat16_rn(a);
            d[i] = h;
            if (MODE == 2) d[i + lo_off] = __float2bfloat16_rn(a - __bfloat162float(h));
        }
    }
}

// The same batch as a BACKGROUND kernel (queued passes: the casts of pass i+1 run while the fused kernel of pass i owns the
// tensor cores).  It has to fit beside a resident CTA of the persistent fused kernel (640 threads x 96 registers, ~183 KB of
// shared memory): ONE CTA per SM of 128 threads x <= 32 registers and 40 KB of shared memory.  The bytes in flight that an
// HBM-bound copy needs therefore live in shared memory, not in registers: every warp keeps kBgStages bulk copies
// (cp.async.bulk, 2 KB of fp64 each, L2 evict-first: the source is read once and must not push the fused kernel's K/V
// tiles out of L2) in flight in a ring of its own -- 40 KB per SM -- converts a landed chunk and stores it with 128-byte
// coalesced stores.  No CTA-wide barrier in the loop: beside the fused kernel the four warps are scheduled when its warps
// leave issue slots, each on its own.
constexpr int kBgThreads = 128;
constexpr int kBgChunkUnits = 128;                       // 2-element units per chunk = 2 KB of fp64, 4 units per lane
constexpr int kBgMaxStages = 5;                          // per WARP: every warp runs its own ring (no CTA-wide barrier in the loop)
constexpr int kBgWarps = kBgThreads / 32;
inline size_t bg_smem_bytes(int stages) { return (size_t)kBgWarps * stages * kBgChunkUnits * 16 + (size_t)kBgWarps * kBgMaxStages * 8; }
// ring depth per warp (SDPA_BG_STAGES, 1..5; default 2 = 16 KB of shared memory per CTA: measured on c3 beside the fused
// kernel, 1 / 2 / 3 / 5 stages give the same step, 217.3 / 216.9 / 219.0 / 216.5 us -- the cast has 190 us to hide in)
inline int bg_stages()
{
    static const int st = [] {
        const char* e = getenv("SDPA_BG_STAGES");
        const int v = e ? atoi(e) : 2;
        return v < 1 ? 1 : (v > kBgMaxStages ? kBgMaxStages : v);
    }();
    return st;
}

__device__ __forceinline__ void bulk_load_evict_first(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar)
{
    uint64_t policy;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(policy));
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;"
                 :: "r"(umma::smem_u32(smem_dst)), "l"(gsrc), "r"(bytes), "r"(umma::smem_u32(bar)), "l"(policy) : "memory");
}

__device__ __forceinline__ unsigned long long cast_global_ns()
{
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
__global__ void stamp_kernel(unsigned long long* dst) { *dst = cast_global_ns(); }

template <int MODE>
__global__ void __launch_bounds__(kBgThreads, 16) cvt_in_batch_bg_kernel(CastBatch cb, int kBgStages, int streaming_stores)
{
    extern __shared__ __align__(128) uint8_t bg_smem[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (cb.trace && threadIdx.x == 0) cb.trace[2 * blockIdx.x] = cast_global_ns();
    double2* ring = reinterpret_cast<double2*>(bg_smem) + (size_t)warp * kBgStages * kBgChunkUnits;
    uint64_t* full = reinterpret_cast<uint64_t*>(bg_smem + (size_t)kBgWarps * kBgStages * kBgChunkUnits * 16) + warp * kBgMaxStages;
    // chunks: segment after segment, every segment's last chunk may be short; warp w of CTA c takes chunks c*4+w, +4*grid, ...
    const unsigned int c0 = (unsigned int)((cb.units[0] + kBgChunkUnits - 1) / kBgChunkUnits);
    const unsigned int c1 = c0 + (unsigned int)((cb.units[1] + kBgChunkUnits - 1) / kBgChunkUnits);
    const unsigned int nchunks = c1 + (unsigned int)((cb.units[2] + kBgChunkUnits - 1) / kBgChunkUnits);
    const unsigned int first_chunk = blockIdx.x * kBgWarps + warp, stride = gridDim.x * kBgWarps;
    auto locate = [&](unsigned int chunk, int& seg, size_t& first, unsigned int& units) {
        seg = chunk < c0 ? 0 : (chunk < c1 ? 1 : 2);
        first = (size_t)(chunk - (seg == 0 ? 0u : (seg == 1 ? c0 : c1))) * kBgChunkUnits;
        const size_t left = cb.units[seg] - first;
        units = left < (size_t)kBgChunkUnits ? (unsigned int)left : (unsigned int)kBgChunkUnits;
    };
    auto issue = [&](unsigned int chunk, int stage) {
        int seg;
        size_t first;
        unsigned int units;
        locate(chunk, seg, first, units);
        umma::mbar_arrive_expect_tx(&full[stage], units * 16u);
        bulk_load_evict_first(ring + (size_t)stage * kBgChunkUnits, reinterpret_cast<const double2*>(cb.src[seg]) + first, units * 16u, &full[stage]);
    };
    if (lane == 0) {
        for (int st = 0; st < kBgStages; ++st) umma::mbar_init(&full[st], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        for (int st = 0; st < kBgStages; ++st) {
            const unsigned int chunk = first_chunk + (unsigned int)st * stride;
            if (chunk < nchunks) issue(chunk, st);
        }
    }
    __syncwarp();
    unsigned int k = 0;
    for (unsigned int chunk = first_chunk; chunk < nchunks; chunk += stride, ++k) {
        const int stage = (int)(k % kBgStages);
        int seg;
        size_t first;
        unsigned int units;
        locate(chunk, seg, first, units);
        umma::mbar_wait(&full[stage], (k / kBgStages) & 1u, 90);
        const double2* in = ring + (size_t)stage * kBgChunkUnits;
        void* dst = cb.dst[seg];
        const size_t lo = cb.lo_off[seg];
        double2 v[kBgChunkUnits / 32];
#pragma unroll
        for (int j = 0; j < kBgChunkUnits / 32; ++j) v[j] = in[j * 32 + lane];
#pragma unroll
        for (int j = 0; j < kBgChunkUnits / 32; ++j) {
            const unsigned int u = j * 32 + lane;
            if (u >= units) continue;
            const size_t off = first + u;
            // streaming_stores: the converted operands belong to the NEXT pass -- stored evict-first they do not push the running
            // fused kernel's K/V tiles out of L2
            if (MODE == 2) {
                uint32_t h, l;
                split_bf16x2(v[j], h, l);
                if (streaming_stores) {
                    __stcs(reinterpret_cast<unsigned int*>(dst) + off, h);
                    __stcs(reinterpret_cast<unsigned int*>(dst) + off + lo, l);
                } else {
                    reinterpret_cast<uint32_t*>(dst)[off] = h;
                    reinterpret_cast<uint32_t*>(dst)[off + lo] = l;
                }
            } else if (MODE == 1) {
                const uint32_t w = pack_bf16x2(__double2float_rn(v[j].x), __double2float_rn(v[j].y));
                if (streaming_stores) __stcs(reinterpret_cast<unsigned int*>(dst) + off, w);
                else reinterpret_cast<uint32_t*>(dst)[off] = w;
            } else {
                const float2 w = make_float2(__double2float_rn(v[j].x), __double2float_rn(v[j].y));
                if (streaming_stores) __stcs(reinterpret_cast<float2*>(dst) + off, w);
                else reinterpret_cast<float2*>(dst)[off] = w;
            }
        }
        __syncwarp();   // every lane has read its share of the stage
        const unsigned int next = chunk + (unsigned int)kBgStages * stride;
        if (lane == 0 && next < nchunks) issue(next, stage);
    }
    if (cb.trace) {
        __syncthreads();
        if (threadIdx.x == 0) cb.trace[2 * blockIdx.x + 1] = cast_global_ns();
    }
}

inline int cast_grid(size_t work_items)
{
    // 148 SMs x 8 resident CTAs of 256 threads; never more CTAs than work.
    const size_t want = (work_items + kCastThreads - 1) / kCastThreads;
    const size_t cap = 148 * 8;
    size_t g = want < cap ? want : cap;
    return (int)(g == 0 ? 1 : g);
}

inline bool aligned(const void* p, size_t a) { return ((uintptr_t)p % a) == 0; }

}  // namespace

static unsigned long long* g_cast_trace = nullptr;
void set_cast_trace(unsigned long long* buf) { g_cast_trace = buf; }
sdpa_status launch_stamp(unsigned long long* dst, cudaStream_t stream)
{
    stamp_kernel<<<1, 1, 0, stream>>>(dst);
    SDPA_CUDA_TRY(cudaGetLastError());
    return SDPA_OK;
}

void preload_cast_kernels()
{
    cudaFuncAttributes a;
    cudaFuncGetAttributes(&a, cvt_in_batch_kernel<double, 0>);
    cudaFuncGetAttributes(&a, cvt_in_batch_kernel<double, 1>);
    cudaFuncGetAttributes(&a, cvt_in_batch_kernel<double, 2>);
    cudaFuncGetAttributes(&a, cvt_in_batch_bg_kernel<0>);
    cudaFuncGetAttributes(&a, cvt_in_batch_bg_kernel<1>);
    cudaFuncGetAttributes(&a, cvt_in_batch_bg_kernel<2>);
    cudaFuncGetAttributes(&a, cvt_d2f_vec_kernel);
    cudaFuncGetAttributes(&a, cvt_d2bf16_vec_kernel);
    cudaFuncGetAttributes(&a, cvt_d2bf16x2_vec_kernel);
    cudaFuncGetAttributes(&a, cvt_f2d_vec_kernel);
    cudaGetLastError();
}

sdpa_status launch_cvt_d2f(float* dst, const double* src, size_t count, cudaStream_t stream)
{
    if (count == 0) return SDPA_OK;
    size_t done = 0;
    if (aligned(dst, 8) && aligned(src, 16) && count >= 2) {
        const size_t units = count / 2;
        cvt_d2f_vec_kernel<<<cast_grid(units / kUnroll), kCastThreads, 0, stream>>>(
            reinterpret_cast<float2*>(dst), reinterpret_cast<const double2*>(src), units);
        count_launch();
        done = units * 2;
    }
    if (done < count) {
        cvt_d2f_scalar_kernel<<<cast_grid(count - done), kCastThreads, 0, stream>>>(dst, src, done, count);
        count_launch();
    }
    SDPA_CUDA_TRY(cudaGetLastError());
    return SDPA_OK;
}

sdpa_status launch_cvt_f2d(double* dst, const float* src, size_t count, cudaStream_t stream)
{
    if (count == 0) return SDPA_OK;
    size_t done = 0;
    if (aligned(dst, 16) && aligned(src, 16) && count >= 4) {
        const size_t units = count / 4;
        cvt_f2d_vec_kernel<<<cast_grid(units / kUnroll), kCastThreads, 0, stream>>>(
            reinterpret_cast<double2*>(dst), reinterpret_cast<const float4*>(src), units);
        count_launch();
        done = units * 4;
    }
    if (done < count) {
        cvt_f2d_scalar_kernel<<<cast_grid(count - done), kCastThreads, 0, stream>>>(dst, src, done, count);
        count_launch();
    }
    SDPA_CUDA_TRY(cudaGetLastError());
    return SDPA_OK;
}

sdpa_status launch_cvt_d2bf16(__nv_bfloat16* dst, const double* src, size_t count, cudaStream_t stream)
{
    if (count == 0) return SDPA_OK;
    size_t done = 0;
    if (aligned(dst, 4) && aligned(src, 16) && count >= 2) {
        const size_t units = count / 2;
        cvt_d2bf16_vec_kernel<<<cast_grid(units / kUnroll), kCastThreads, 0, stream>>>(
            reinterpret_cast<uint32_t*>(dst), reinterpret_cast<const double2*>(src), units);
        count_launch();
        done = units * 2;
    }
    if (done < count) {
        cvt_d2bf16_scalar_kernel<<<cast_grid(count - done), kCastThreads, 0, stream>>>(dst, src, done, count);
        count_launch();
    }
    SDPA_CUDA_TRY(cudaGetLastError());
    return SDPA_OK;
}

sdpa_status launch_cvt_d2bf16x2(__nv_bfloat16* dst_hi, __nv_bfloat16* dst_lo, const double* src, size_t count, cudaStream_t stream)
{
    if (count == 0) return SDPA_OK;
    size_t done = 0;
    if (aligned(dst_hi, 4) && aligned(dst_lo, 4) && aligned(src, 16) && count >= 2) {
        const size_t units = count / 2;
        cvt_d2bf16x2_vec_kernel<<<cast_grid(units / kUnroll), kCastThreads, 0, stream>>>(
            reinterpret_cast<uint32_t*>(dst_hi), reinterpret_cast<uint32_t*>(dst_lo), reinterpret_cast<const double2*>(src), units);
        count_launch();
        done = units * 2;
    }
    if (done < count) {
        cvt_d2bf16x2_scalar_kernel<<<cast_grid(count - done), kCastThreads, 0, stream>>>(dst_hi, dst_lo, src, done, count);
        count_launch();
    }
    SDPA_CUDA_TRY(cudaGetLastError());
    return SDPA_OK;
}

template <typename SRC>
static void launch_in_batch(int prec, const CastBatch& cb, int grid, cudaStream_t stream)
{
    if (prec == SDPA_PREC_BF16X3) cvt_in_batch_kernel<SRC, 2><<<grid, kCastThreads, 0, stream>>>(cb);
    else if (prec == SDPA_PREC_BF16) cvt_in_batch_kernel<SRC, 1><<<grid, kCastThreads, 0, stream>>>(cb);
    else cvt_in_batch_kernel<SRC, 0><<<grid, kCastThreads, 0, stream>>>(cb);
}
template <typename SRC>
static void launch_typed_scalar(int prec, void* dst, size_t lo_off, const void* src, size_t count, cudaStream_t stream)
{
    const SRC* s = reinterpret_cast<const SRC*>(src);
    if (prec == SDPA_PREC_BF16X3) cvt_typed_scalar_kernel<SRC, 2><<<cast_grid(count), kCastThreads, 0, stream>>>(dst, lo_off, s, count);
    else if (prec == SDPA_PREC_BF16) cvt_typed_scalar_kernel<SRC, 1><<<cast_grid(count), kCastThreads, 0, stream>>>(dst, lo_off, s, count);
    else cvt_typed_scalar_kernel<SRC, 0><<<cast_grid(count), kCastThreads, 0, stream>>>(dst, lo_off, s, count);
}

// Up to three operands in one launch; falls back to one launch per operand when a pointer is not aligned to a 2-element unit
// (16 B for fp64 sources) or a count is odd (the batched kernel moves 2-element units only).
sdpa_status launch_cvt_in_batch(int src_dtype, int prec, void* const* dst, const void* const* src, const size_t* count,
                                const size_t* lo_off, int nseg, cudaStream_t stream, int background_ctas)
{
    if (nseg < 0 || nseg > 3) {
        set_error("launch_cvt_in_batch: 0..3 segments");
        return SDPA_ERR_INVALID;
    }
    if (src_dtype != SDPA_DTYPE_F64 && src_dtype != SDPA_DTYPE_F32 && src_dtype != SDPA_DTYPE_BF16) {
        set_error("launch_cvt_in_batch: unknown source dtype %d", src_dtype);
        return SDPA_ERR_INVALID;
    }
    if (src_dtype != SDPA_DTYPE_F64 && background_ctas > 0) {   // typed passes never cast ahead
        set_error("launch_cvt_in_batch: the background form takes fp64 sources only");
        return SDPA_ERR_INVALID;
    }
    const size_t src_unit = src_dtype == SDPA_DTYPE_F64 ? 16 : (src_dtype == SDPA_DTYPE_F32 ? 8 : 4);
    bool vec_ok = true;
    size_t units_total = 0;
    CastBatch cb;
    for (int k = 0; k < 3; ++k) {
        cb.dst[k] = nullptr;
        cb.src[k] = nullptr;
        cb.units[k] = 0;
        cb.lo_off[k] = 0;
    }
    cb.trace = background_ctas > 0 ? g_cast_trace : nullptr;
    const bool split = prec == SDPA_PREC_BF16X3;
    for (int k = 0; k < nseg; ++k) {
        if (count[k] == 0) continue;
        vec_ok = vec_ok && (count[k] % 2 == 0) && aligned(src[k], src_unit) && aligned(dst[k], 8) && (!split || (lo_off && lo_off[k] % 2 == 0));
        cb.dst[k] = dst[k];
        cb.src[k] = src[k];
        cb.units[k] = count[k] / 2;
        cb.lo_off[k] = split && lo_off ? lo_off[k] / 2 : 0;
        units_total += cb.units[k];
    }
    if (units_total == 0 && vec_ok) return SDPA_OK;
    if (!vec_ok) {
        for (int k = 0; k < nseg; ++k) {
            if (src_dtype != SDPA_DTYPE_F64) {
                if (count[k] == 0) continue;
                const size_t lo = split && lo_off ? lo_off[k] : 0;
                if (src_dtype == SDPA_DTYPE_F32) launch_typed_scalar<float>(prec, dst[k], lo, src[k], count[k], stream);
                else launch_typed_scalar<__nv_bfloat16>(prec, dst[k], lo, src[k], count[k], stream);
                count_launch();
                SDPA_CUDA_TRY(cudaGetLastError());
                continue;
            }
            const double* s = reinterpret_cast<const double*>(src[k]);
            if (split) {
                __nv_bfloat16* hi = reinterpret_cast<__nv_bfloat16*>(dst[k]);
                SDPA_TRY(launch_cvt_d2bf16x2(hi, hi + (lo_off ? lo_off[k] : 0), s, count[k], stream));
            } else if (prec == SDPA_PREC_BF16) SDPA_TRY(launch_cvt_d2bf16(reinterpret_cast<__nv_bfloat16*>(dst[k]), s, count[k], stream));
            else SDPA_TRY(launch_cvt_d2f(reinterpret_cast<float*>(dst[k]), s, count[k], stream));
        }
        return SDPA_OK;
    }
    if (background_ctas > 0) {
        // small-footprint form, one CTA per SM; same (maximum) shared-memory carveout as the fused kernel it runs beside
        static bool carve_done[64] = {};
        int dev = 0;
        cudaGetDevice(&dev);
        if (dev >= 0 && dev < 64 && !carve_done[dev]) {
            cudaFuncSetAttribute(cvt_in_batch_bg_kernel<0>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
            cudaFuncSetAttribute(cvt_in_batch_bg_kernel<1>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
            cudaFuncSetAttribute(cvt_in_batch_bg_kernel<2>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
            carve_done[dev] = true;
        }
        const int stages = bg_stages();
        const size_t smem = bg_smem_bytes(stages);
        static const int cs = [] {
            const char* e = getenv("SDPA_BG_STORE");   // cs (evict-first stores) | default
            return (e && !strcmp(e, "cs")) ? 1 : 0;
        }();
        if (split) cvt_in_batch_bg_kernel<2><<<background_ctas, kBgThreads, smem, stream>>>(cb, stages, cs);
        else if (prec == SDPA_PREC_BF16) cvt_in_batch_bg_kernel<1><<<background_ctas, kBgThreads, smem, stream>>>(cb, stages, cs);
        else cvt_in_batch_bg_kernel<0><<<background_ctas, kBgThreads, smem, stream>>>(cb, stages, cs);
        count_launch();
        SDPA_CUDA_TRY(cudaGetLastError());
        return SDPA_OK;
    }
    const int grid = cast_grid(units_total / kUnroll);
    if (src_dtype == SDPA_DTYPE_F64) launch_in_batch<double>(prec, cb, grid, stream);
    else if (src_dtype == SDPA_DTYPE_F32) launch_in_batch<float>(prec, cb, grid, stream);
    else launch_in_batch<__nv_bfloat16>(prec, cb, grid, stream);
    count_launch();
    SDPA_CUDA_TRY(cudaGetLastError());
    return SDPA_OK;
}

}  // namespace sdpa
