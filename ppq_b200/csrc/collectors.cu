// collectors.cu -- sm_100a calibration collectors behind the C ABI of include/ppq_b200.h.
//
//   ppq_b200_minmax_t / _c          fused single-pass min+max; replaces the two torch reductions of
//                                   TorchMinMaxObserver.observe (/root/reference/ppq/quantization/observer/range.py:85-100)
//   ppq_b200_histogram_t            replaces Histogram_T            (ppq/csrc/cuda/sort.cu:75-111)
//   ppq_b200_histogram_asym_t       replaces Histogram_Asymmetric_T (sort.cu:113-165)
//   ppq_b200_histogram_c            replaces Histogram_C            (sort.cu:167-218)
//   ppq_b200_multi_*                one launch over a table of tensors (the calibration arena path, DESIGN.md)
//
// All of them read each element exactly once (4 B/element algorithmic traffic) with 128-bit streaming loads, four per
// thread in flight (the multi-tensor min/max and histogram: 256-bit loads, see stream_v8).  Histograms are privatised per CTA in shared memory (bins x int32, 16 KB for the KL observer's 4096
// bins) and counted with an unconditional red.shared.add into `bins + 1` slots (the extra one is a trash slot for dropped
// samples; ptxas emits ATOMS.POPC.INC, which aggregates same-address lanes in hardware, so the post-ReLU pile-up in bin 0 is
// not a hot spot); only non-empty bins are flushed to the caller's global histogram with red.global.add.
#include "common.cuh"
#include "../../include/ppq_b200.h"
#include "variants.h"
#include <cooperative_groups.h>

namespace ppqb {
namespace cg = cooperative_groups;

constexpr int kThreads = 256;
constexpr int kUnroll = 4;

__device__ __forceinline__ float min_nan(float a, float b) { float r; asm("min.NaN.f32 %0, %1, %2;" : "=f"(r) : "f"(a), "f"(b)); return r; }
__device__ __forceinline__ float max_nan(float a, float b) { float r; asm("max.NaN.f32 %0, %1, %2;" : "=f"(r) : "f"(a), "f"(b)); return r; }

// NaN-propagating (min, max) of a thread's values -> warp -> CTA; result valid in thread 0.
struct MinMax {
    float lo, hi;
    __device__ __forceinline__ MinMax() { lo = __int_as_float(0x7F800000); hi = __int_as_float(0xFF800000); }
    __device__ __forceinline__ void add(float v) { lo = min_nan(lo, v); hi = max_nan(hi, v); }
    __device__ __forceinline__ void add4(const float4 &v) { add(v.x); add(v.y); add(v.z); add(v.w); }
    __device__ __forceinline__ void warp_reduce() {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            lo = min_nan(lo, __shfl_xor_sync(0xffffffffu, lo, o));
            hi = max_nan(hi, __shfl_xor_sync(0xffffffffu, hi, o));
        }
    }
    // publish into accumulating global slots (see common.cuh: raw-bit float atomics, NaN poisons both slots)
    __device__ __forceinline__ void publish(float *gmin, float *gmax) const {
        if (lo != lo || hi != hi) {
            atomic_min_float(gmin, __uint_as_float(0xFFC00000u));
            atomic_max_float(gmax, __uint_as_float(0x7FC00000u));
        } else {
            atomic_min_float(gmin, lo);
            atomic_max_float(gmax, hi);
        }
    }
};

__device__ __forceinline__ void block_reduce_publish(MinMax mm, float *gmin, float *gmax) {
    __shared__ float s_lo[kThreads / 32], s_hi[kThreads / 32];
    mm.warp_reduce();
    const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
    if (l == 0) { s_lo[w] = mm.lo; s_hi[w] = mm.hi; }
    __syncthreads();
    if (w == 0) {
        MinMax t;
        if (l < kThreads / 32) { t.lo = s_lo[l]; t.hi = s_hi[l]; }
        t.warp_reduce();
        if (l == 0) t.publish(gmin, gmax);
    }
    __syncthreads();
}

// Streams elements [0, n) of x through `f(float)`; float4 path when the base is 16-byte aligned.
// `first`/`stride` are in units of threads over the whole cooperating group (a grid or a sub-grid).
template <class F>
__device__ __forceinline__ void stream_elements(const float *__restrict__ x, int64_t n, int64_t first, int64_t stride, F &&f) {
    if ((reinterpret_cast<uintptr_t>(x) & 15u) == 0) {
        const int64_t n4 = n >> 2;
        const float4 *x4 = reinterpret_cast<const float4 *>(x);
        // warp-contiguous segments of 32 x kUnroll vectors (lane-interleaved): a thread's kUnroll loads in flight fall into one 2 KB
        // span of HBM (same pattern as the fake-quant kernels, where it measured +3..4 points of HBM peak over grid-stride)
        constexpr int64_t kSeg = 32 * kUnroll;
        const int64_t lane = first & 31, warp = first >> 5, warps = stride >> 5;
        const int64_t segs = (n4 + kSeg - 1) / kSeg;
        for (int64_t sg = warp; sg < segs; sg += warps) {
            const int64_t base = sg * kSeg + lane;
            float4 v[kUnroll];
#pragma unroll
            for (int j = 0; j < kUnroll; j++) if (base + j * 32 < n4) v[j] = ld_stream4(x4 + base + j * 32);
#pragma unroll
            for (int j = 0; j < kUnroll; j++) if (base + j * 32 < n4) { f(v[j].x); f(v[j].y); f(v[j].z); f(v[j].w); }
        }
        const int64_t t = (n4 << 2) + first;
        if (t < n) f(x[t]);
    } else {
        for (int64_t i = first; i < n; i += stride) f(ld_stream1(x + i));
    }
}

// ---- min / max ------------------------------------------------------------------------------------------------------
__global__ void minmax_init_kernel(float *mins, float *maxs, int64_t count) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < count) {
        if (mins) mins[i] = __int_as_float(0x7F800000);
        if (maxs) maxs[i] = __int_as_float(0xFF800000);
    }
}

__global__ void __launch_bounds__(kThreads)
minmax_t_kernel(const float *__restrict__ x, int64_t n, float *__restrict__ minmax) {
    MinMax mm;
    stream_elements(x, n, (int64_t)blockIdx.x * kThreads + threadIdx.x, (int64_t)gridDim.x * kThreads,
                    [&](float v) { mm.add(v); });
    block_reduce_publish(mm, minmax, minmax + 1);
}

// One tensor per descriptor, work item = (tensor, chunk of `chunk` elements); blockIdx.x walks the items.
__global__ void __launch_bounds__(kThreads)
multi_minmax_t_kernel(const ppq_b200_tensor_desc *__restrict__ descs, int count, int64_t chunk, int chunks_per_tensor,
                      float *__restrict__ arena) {
    const int64_t items = (int64_t)count * chunks_per_tensor;
    for (int64_t item = blockIdx.x; item < items; item += gridDim.x) {
        const int t = (int)(item / chunks_per_tensor);
        const int64_t c = item - (int64_t)t * chunks_per_tensor;
        const ppq_b200_tensor_desc d = descs[t];
        const int64_t begin = c * chunk;
        if (begin >= d.n) continue;                                    // uniform per CTA
        const int64_t len = (d.n - begin) < chunk ? (d.n - begin) : chunk;
        MinMax mm;
        stream_elements(d.x + begin, len, threadIdx.x, kThreads, [&](float v) { mm.add(v); });
        block_reduce_publish(mm, arena + 2 * (int64_t)d.slot, arena + 2 * (int64_t)d.slot + 1);
    }
}

// Per channel: tensor = rows x epc, channel(row) = row % C.  One warp per (row, chunk) work item.
constexpr int kRowChunk = 4096;
__global__ void __launch_bounds__(kThreads)
minmax_c_kernel(const float *__restrict__ x, int64_t rows, int64_t epc, int C, int64_t chunks_per_row,
                FastDiv div_chunks, FastDiv div_C, float *__restrict__ mins, float *__restrict__ maxs) {
    const int lane = threadIdx.x & 31;
    const int64_t warps = (int64_t)gridDim.x * (kThreads / 32);
    const int64_t items = rows * chunks_per_row;
    for (int64_t item = (int64_t)blockIdx.x * (kThreads / 32) + (threadIdx.x >> 5); item < items; item += warps) {
        const int64_t row = (int64_t)div_chunks.quot((uint64_t)item);
        const int64_t chunk = item - row * chunks_per_row;
        const int c = (int)(row - (int64_t)div_C.quot((uint64_t)row) * C);
        const int64_t begin = chunk * kRowChunk;
        const int64_t len = (epc - begin) < kRowChunk ? (epc - begin) : kRowChunk;
        MinMax mm;
        stream_elements(x + row * epc + begin, len, lane, 32, [&](float v) { mm.add(v); });
        mm.warp_reduce();
        if (lane == 0) mm.publish(mins + c, maxs + c);
    }
}

// ---- histograms -------------------------------------------------------------------------------------------------------
// Binning operators map a value to a slot of the CTA-private shared histogram: slots 0..bins-1 are the bins, slot `bins`
// is a trash slot for dropped samples, so that the shared atomic is unconditional (no branch per element; ptxas turns
// `red.shared.add.u32 [a], 1` into ATOMS.POPC.INC, which aggregates same-address lanes of a warp in hardware -- the
// post-ReLU pile-up in bin 0 costs one pass, not 32).
struct BinParams { float a, b; int bins, clip; };   // sym: a = hist_scale;  asym: a = min, b = max
struct SymBin {
    ExactDiv d; unsigned bins; int last; bool clip;
    __device__ __forceinline__ SymBin(float hist_scale, int nbins, bool clip_outliers) : bins(nbins), last(nbins - 1), clip(clip_outliers) { d.init(hist_scale); }
    __device__ __forceinline__ explicit SymBin(const BinParams &p) : SymBin(p.a, p.bins, p.clip != 0) {}
    __device__ __forceinline__ unsigned finish(float t) const {
        const int b = __float2int_rd(t);                              // (int) floor(.), saturating, NaN -> 0; never negative here
        return clip ? min((unsigned)b, bins) : (unsigned)min(b, last);
    }
    __device__ __forceinline__ unsigned operator()(float v) const { return finish(d.div(fabsf(v))); }
    __device__ __forceinline__ uint4 bin4(const float4 &v) const {
        const float4 t = d.div4(make_float4(fabsf(v.x), fabsf(v.y), fabsf(v.z), fabsf(v.w)));
        return make_uint4(finish(t.x), finish(t.y), finish(t.z), finish(t.w));
    }
};
struct AsymBin {
    ExactDiv d; float vmin; unsigned bins; int last; bool clip;
    __device__ __forceinline__ AsymBin(float mn, float mx, int nbins, bool clip_outliers) : vmin(mn), bins(nbins), last(nbins - 1), clip(clip_outliers) {
        d.init(__fdiv_rn(__fsub_rn(mx, mn), (float)nbins));           // hist_scale = (max - min) / bins, in fp32
    }
    __device__ __forceinline__ explicit AsymBin(const BinParams &p) : AsymBin(p.a, p.b, p.bins, p.clip != 0) {}
    __device__ __forceinline__ unsigned finish(float t) const {
        const int b = __float2int_rd(t);
        return clip ? min((unsigned)b, bins) : (unsigned)max(min(b, last), 0);   // negative b wraps above `bins` -> trash
    }
    __device__ __forceinline__ unsigned operator()(float v) const { return finish(d.div(__fsub_rn(v, vmin))); }
    __device__ __forceinline__ uint4 bin4(const float4 &v) const {
        const float4 t = d.div4(make_float4(__fsub_rn(v.x, vmin), __fsub_rn(v.y, vmin), __fsub_rn(v.z, vmin), __fsub_rn(v.w, vmin)));
        return make_uint4(finish(t.x), finish(t.y), finish(t.z), finish(t.w));
    }
};

// Counting into the CTA-private histogram.
//   VARIANT 0 (default): unconditional red.shared.add through a precomputed 32-bit shared-window address.
//   VARIANT 1: the same through generic-pointer atomicAdd;  VARIANT 2: __match_any_sync aggregation in software;
//   VARIANT 3: global atomics straight into `hist` (what the reference does; kept for A/B measurements only).
template <int VARIANT>
struct Counter {
    int *sh; int32_t *gh; uint32_t sh_addr; unsigned trash;
    __device__ __forceinline__ Counter(int *smem_hist, int32_t *global_hist, int bins)
        : sh(smem_hist), gh(global_hist), sh_addr((uint32_t)__cvta_generic_to_shared(smem_hist)), trash(bins) {}
    __device__ __forceinline__ void count(unsigned slot) {
        if constexpr (VARIANT == 0) {
            asm volatile("red.shared.add.u32 [%0], 1;" ::"r"(sh_addr + slot * 4u) : "memory");
        } else if constexpr (VARIANT == 1) {
            atomicAdd(sh + slot, 1);
        } else if constexpr (VARIANT == 2) {
            const unsigned peers = __match_any_sync(0xffffffffu, slot);
            if ((threadIdx.x & 31) == (__ffs(peers) - 1)) atomicAdd(sh + slot, __popc(peers));
        } else {
            if (slot != trash) atomicAdd(gh + slot, 1);
        }
    }
};

template <int VARIANT>
__device__ __forceinline__ void hist_zero(int *sh, int bins) {
    if constexpr (VARIANT != 3) {
        for (int i = threadIdx.x; i <= bins; i += blockDim.x) sh[i] = 0;    // + the trash slot
        __syncthreads();
    }
}
template <int VARIANT>
__device__ __forceinline__ void hist_flush(const int *sh, int bins, int32_t *gh) {
    if constexpr (VARIANT != 3) {
        __syncthreads();
        for (int i = threadIdx.x; i < bins; i += blockDim.x) {
            const int v = sh[i];
            if (v) atomicAdd(gh + i, v);
        }
        __syncthreads();
    }
}

// The ballot in VARIANT 0/2 needs all 32 lanes of a warp to call count() the same number of times: stream_elements
// gives every lane of a warp the same trip count except in the ragged tail, so tails are padded with "drop" (-1).
template <int VARIANT, class Bin, int U = kUnroll>
__device__ __forceinline__ void hist_stream(const float *__restrict__ x, int64_t n, int64_t first, int64_t stride,
                                            const Bin &bin, Counter<VARIANT> &cnt) {
    if ((reinterpret_cast<uintptr_t>(x) & 15u) == 0) {
        const int64_t n4 = n >> 2;
        const float4 *x4 = reinterpret_cast<const float4 *>(x);
        const int64_t warp_first = first - (threadIdx.x & 31);              // lane 0 of this warp
        int64_t i = first;
        // full unrolled rounds: uniform across the warp because lanes are consecutive in i
        for (; warp_first + (i - first) + 31 + (U - 1) * stride < n4; i += U * stride) {
            float4 v[U];
#pragma unroll
            for (int j = 0; j < U; j++) v[j] = ld_stream4(x4 + i + j * stride);
#pragma unroll
            for (int j = 0; j < U; j++) { const uint4 b = bin.bin4(v[j]); cnt.count(b.x); cnt.count(b.y); cnt.count(b.z); cnt.count(b.w); }
        }
        // remaining rounds: warp-uniform loop bound, per-lane predicate
        for (; warp_first + (i - first) < n4; i += stride) {
            const bool ok = i < n4;
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (ok) v = ld_stream4(x4 + i);
            const uint4 b = bin.bin4(v);
            cnt.count(ok ? b.x : cnt.trash); cnt.count(ok ? b.y : cnt.trash); cnt.count(ok ? b.z : cnt.trash); cnt.count(ok ? b.w : cnt.trash);
        }
        const int64_t t = (n4 << 2) + first;
        const bool tail_any = (n4 << 2) + warp_first < n;                    // warp-uniform
        if (tail_any) cnt.count(t < n ? bin(x[t]) : cnt.trash);
    } else {
        const int64_t warp_first = first - (threadIdx.x & 31);
        for (int64_t i = first; warp_first + (i - first) < n; i += stride) cnt.count(i < n ? bin(ld_stream1(x + i)) : cnt.trash);
    }
}

constexpr int kHistThreads = 1024;   // big CTAs: the flush of the private bins (bins global atomics per CTA) is what limits small-CTA
                                     // configurations (measured: 256 thr x 8/SM 59 % -> 1024 thr x 1/SM 82-86 % -> 1024 thr x 2/SM, two
                                     // loads in flight, 87 % of HBM peak: r02_kbench.txt)
template <int VARIANT, class Bin, int U = kUnroll, int TPB = kHistThreads, int MINB = 1>
__global__ void __launch_bounds__(TPB, MINB)
histogram_kernel(const float *__restrict__ x, int64_t n, BinParams bp, int32_t *__restrict__ hist) {
    extern __shared__ int sh[];
    const int bins = bp.bins;
    hist_zero<VARIANT>(sh, bins);
    Counter<VARIANT> cnt(sh, hist, bins);
    const Bin bin(bp);
    hist_stream<VARIANT, Bin, U>(x, n, (int64_t)blockIdx.x * TPB + threadIdx.x, (int64_t)gridDim.x * TPB, bin, cnt);
    hist_flush<VARIANT>(sh, bins, hist);
}

// Cluster variant (A/B: variants 7 / 8 = clusters of 2 / 4 CTAs): the CTAs of a thread-block cluster reduce their private bins through
// distributed shared memory before touching global memory -- CTA r sums slice r of all CL private histograms with DSMEM loads and flushes
// only that slice, so a launch issues grid / CL x bins global atomics instead of grid x bins (the flush of 148 x 4096 counters is the fixed
// cost that separates the single-tensor collector from the multi-tensor one, DESIGN.md §5).
template <class Bin, int CL>
__global__ void __cluster_dims__(CL, 1, 1) __launch_bounds__(kHistThreads)
histogram_cluster_kernel(const float *__restrict__ x, int64_t n, BinParams bp, int32_t *__restrict__ hist) {
    extern __shared__ int sh[];
    cg::cluster_group cluster = cg::this_cluster();
    const int bins = bp.bins;
    hist_zero<0>(sh, bins);
    Counter<0> cnt(sh, hist, bins);
    const Bin bin(bp);
    hist_stream<0, Bin>(x, n, (int64_t)blockIdx.x * kHistThreads + threadIdx.x, (int64_t)gridDim.x * kHistThreads, bin, cnt);
    cluster.sync();                                                     // every CTA of the cluster has finished counting
    const unsigned r = cluster.block_rank();
    const int *peer[CL];
#pragma unroll
    for (int c = 0; c < CL; c++) peer[c] = cluster.map_shared_rank(sh, c);
    const int slice = (bins + CL - 1) / CL, b0 = (int)r * slice, b1 = min(bins, b0 + slice);
    for (int i = b0 + (int)threadIdx.x; i < b1; i += kHistThreads) {
        int v = 0;
#pragma unroll
        for (int c = 0; c < CL; c++) v += peer[c][i];
        if (v) atomicAdd(hist + i, v);
    }
    cluster.sync();                                                     // nobody exits while a peer still reads its shared memory
}

// hist_scale read from device memory (phase 2 without a host round trip)
template <int VARIANT>
__global__ void __launch_bounds__(kHistThreads, 2)
histogram_dscale_kernel(const float *__restrict__ x, int64_t n, const float *__restrict__ hist_scale, int clip, int bins,
                        int32_t *__restrict__ hist) {
    extern __shared__ int sh[];
    hist_zero<VARIANT>(sh, bins);
    Counter<VARIANT> cnt(sh, hist, bins);
    const SymBin bin(__ldg(hist_scale), bins, clip != 0);
    hist_stream<VARIANT, SymBin, 2>(x, n, (int64_t)blockIdx.x * kHistThreads + threadIdx.x, (int64_t)gridDim.x * kHistThreads, bin, cnt);
    hist_flush<VARIANT>(sh, bins, hist);
}

template <int VARIANT>
__global__ void __launch_bounds__(kHistThreads)
multi_histogram_t_kernel(const ppq_b200_tensor_desc *__restrict__ descs, int count,
                         const float *__restrict__ hist_scale_arena, int clip, int bins, int32_t *__restrict__ hist_arena) {
    // Each CTA owns one contiguous span of the concatenation of all tensors, so the private bins are zeroed / flushed
    // (#CTAs + #tensors) times in total instead of once per fixed-size chunk.
    extern __shared__ int sh[];
    int64_t *prefix = reinterpret_cast<int64_t *>(sh + ((bins + 1 + 1) & ~1));       // [count + 1], 8-byte aligned
    if (threadIdx.x == 0) {
        int64_t run = 0;
        for (int t = 0; t < count; t++) { prefix[t] = run; run += descs[t].n; }
        prefix[count] = run;
    }
    __syncthreads();
    const int64_t total = prefix[count];
    int64_t span = (total + gridDim.x - 1) / gridDim.x;
    span = (span + 3) & ~(int64_t)3;
    const int64_t s0 = (int64_t)blockIdx.x * span, s1 = (s0 + span) < total ? (s0 + span) : total;
    if (s0 >= total) return;
    int t = 0;                                                         // first tensor overlapping [s0, s1): binary search
    { int lo = 0, hi = count - 1; while (lo < hi) { const int mid = (lo + hi + 1) >> 1; if (prefix[mid] <= s0) lo = mid; else hi = mid - 1; } t = lo; }
    for (; t < count && prefix[t] < s1; t++) {
        const ppq_b200_tensor_desc d = descs[t];
        int64_t a = s0 - prefix[t]; if (a < 0) a = 0;
        int64_t b = s1 - prefix[t]; if (b > d.n) b = d.n;
        a = (a + 3) & ~(int64_t)3; if (a > d.n) a = d.n;               // both neighbours round the shared boundary the same way
        if (b < d.n) b = (b + 3) & ~(int64_t)3; if (b > d.n) b = d.n;
        if (b <= a) continue;                                          // uniform per CTA
        int32_t *gh = hist_arena + (int64_t)d.slot * bins;
        hist_zero<VARIANT>(sh, bins);
        Counter<VARIANT> cnt(sh, gh, bins);
        const SymBin bin(__ldg(hist_scale_arena + d.slot), bins, clip != 0);
        hist_stream<VARIANT>(d.x + a, b - a, threadIdx.x, kHistThreads, bin, cnt);
        hist_flush<VARIANT>(sh, bins, gh);
    }
}

// Per-channel histogram: rows x epc, hist[c][bins].  One CTA per (row, chunk); smem holds that row's private bins.
template <int VARIANT>
__global__ void __launch_bounds__(kThreads)
histogram_c_kernel(const float *__restrict__ x, int64_t rows, int64_t epc, int C, int64_t chunk, int64_t chunks_per_row,
                   float hist_scale, int clip, int bins, int32_t *__restrict__ hist) {
    extern __shared__ int sh[];
    const int64_t items = rows * chunks_per_row;
    const SymBin bin(hist_scale, bins, clip != 0);
    for (int64_t item = blockIdx.x; item < items; item += gridDim.x) {
        const int64_t row = item / chunks_per_row;
        const int64_t c0 = item - row * chunks_per_row;
        const int ch = (int)(row % C);
        const int64_t begin = c0 * chunk;
        const int64_t len = (epc - begin) < chunk ? (epc - begin) : chunk;
        int32_t *gh = hist + (int64_t)ch * bins;
        hist_zero<VARIANT>(sh, bins);
        Counter<VARIANT> cnt(sh, gh, bins);
        hist_stream<VARIANT>(x + row * epc + begin, len, threadIdx.x, kThreads, bin, cnt);
        hist_flush<VARIANT>(sh, bins, gh);
    }
}

// ---- multi-tensor streaming collectors ---------------------------------------------------------------------------------
// The launch reads the concatenation of all tensors once.  Every CTA owns one contiguous span of equal length of that
// concatenation (no empty work items however ragged the table is) and walks the tensors overlapping it; a CTA's statistics
// for one tensor are published once.  Loads are 256-bit (LDG.E.256 on sm_100a), U per thread in flight, lane-interleaved
// inside warp-contiguous segments; the head up to the first 32-byte boundary and the ragged tail go through scalar loads,
// so any 4-byte aligned base is on the vector path.

struct float8v { float4 a, b; };
__device__ __forceinline__ float8v ld_stream8(const float *p) {
    float8v v;
    asm volatile("ld.global.nc.L1::no_allocate.L2::evict_first.L2::256B.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=f"(v.a.x), "=f"(v.a.y), "=f"(v.a.z), "=f"(v.a.w), "=f"(v.b.x), "=f"(v.b.y), "=f"(v.b.z), "=f"(v.b.w) : "l"(p));
    return v;
}

// Elements [0, n) of x, split over `nthreads` threads of the calling CTA: f4(float4) for vector data, f1(float) for the
// head and tail elements.
template <int U, class F4, class F1>
__device__ __forceinline__ void stream_v8(const float *__restrict__ x, int64_t n, int tid, int nthreads, F4 &&f4, F1 &&f1) {
    const int64_t to_boundary = (int64_t)(((32u - ((uint32_t)reinterpret_cast<uintptr_t>(x) & 31u)) & 31u) >> 2);
    const int head = (int)(to_boundary < n ? to_boundary : n);
    if (tid < head) f1(ld_stream1(x + tid));
    x += head; n -= head;
    const float *const end = x + (n & ~(int64_t)7);                    // end of the vector part
    constexpr int kSeg = 32 * 8 * U;                                   // floats per warp segment
    const int64_t step = (int64_t)(nthreads >> 5) * kSeg;
    for (const float *p = x + (int64_t)(tid >> 5) * kSeg + (tid & 31) * 8; p < end; p += step) {
        float8v v[U];
#pragma unroll
        for (int j = 0; j < U; j++) if (p + j * 256 < end) v[j] = ld_stream8(p + j * 256);
#pragma unroll
        for (int j = 0; j < U; j++) if (p + j * 256 < end) { f4(v[j].a); f4(v[j].b); }
    }
    const float *t = end + tid;
    if (t < x + n) f1(ld_stream1(t));
}

// prefix[t] = elements of tensors 0 .. t-1 (prefix[count] = total), built in shared memory by the whole CTA: one parallel
// round of descriptor loads, then a chunked warp scan.
__device__ __forceinline__ int64_t build_prefix(const ppq_b200_tensor_desc *__restrict__ descs, int count, int64_t *prefix) {
    for (int i = threadIdx.x; i < count; i += blockDim.x) { const int64_t n = descs[i].n; prefix[i + 1] = n > 0 ? n : 0; }
    if (threadIdx.x == 0) prefix[0] = 0;
    __syncthreads();
    if (threadIdx.x < 32) {
        const int lane = threadIdx.x;
        int64_t carry = 0;
        for (int b = 1; b <= count; b += 32) {
            const int i = b + lane;
            int64_t v = i <= count ? prefix[i] : 0;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) { const int64_t w = __shfl_up_sync(0xffffffffu, v, o); if (lane >= o) v += w; }
            v += carry;
            if (i <= count) prefix[i] = v;
            carry = __shfl_sync(0xffffffffu, v, 31);
        }
    }
    __syncthreads();
    return prefix[count];
}

// This CTA's span [s0, s1) of the concatenation and the first tensor overlapping it; false when the span is empty.
__device__ __forceinline__ bool cta_span(const int64_t *prefix, int count, int64_t total, int64_t &s0, int64_t &s1, int &t) {
    const int64_t span = (total + gridDim.x - 1) / gridDim.x;
    s0 = (int64_t)blockIdx.x * span;
    s1 = min(s0 + span, total);
    if (s0 >= total) return false;
    int lo = 0, hi = count - 1;                                        // last t with prefix[t] <= s0
    while (lo < hi) { const int mid = (lo + hi + 1) >> 1; if (prefix[mid] <= s0) lo = mid; else hi = mid - 1; }
    t = lo;
    return true;
}

// min/max: each warp folds its share of a (CTA, tensor) piece in registers and publishes it with two atomics, no CTA barrier.
template <int TPB, int MINB, int U>
__global__ void __launch_bounds__(TPB, MINB)
multi_minmax_stream_kernel(const ppq_b200_tensor_desc *__restrict__ descs, int count, float *__restrict__ arena) {
    extern __shared__ int64_t prefix[];
    const int64_t total = build_prefix(descs, count, prefix);
    int64_t s0, s1; int t;
    if (!cta_span(prefix, count, total, s0, s1, t)) return;
    for (; t < count && prefix[t] < s1; t++) {
        const ppq_b200_tensor_desc d = descs[t];
        const int64_t a = max(s0 - prefix[t], (int64_t)0), b = min(s1 - prefix[t], d.n);
        if (b <= a) continue;                                          // uniform per CTA
        MinMax mm;
        stream_v8<U>(d.x + a, b - a, threadIdx.x, TPB, [&](const float4 &v) { mm.add4(v); }, [&](float v) { mm.add(v); });
        mm.warp_reduce();
        const bool empty = mm.lo == __int_as_float(0x7F800000) && mm.hi == __int_as_float(0xFF800000);   // warp saw no element
        if ((threadIdx.x & 31) == 0 && !empty) mm.publish(arena + 2 * (int64_t)d.slot, arena + 2 * (int64_t)d.slot + 1);
    }
}

// SymBin's slot with a full-rate floor: for 0 <= u < 2^23, u + 2^23 rounded down is 2^23 + floor(u), whose bit pattern is
// 0x4B000000 + floor(u).  Clamping the quotient to [0, cap] before the floor gives min(floor(q), cap) as SymBin does
// (cap = bins: the trash slot, or bins - 1), and fmaxf sends a NaN quotient to slot 0 like F2I.  The slot's byte address in
// the shared histogram is folded into one integer multiply-add of the float's bits.
struct SymSlot {
    ExactDiv d; float cap; uint32_t base;
    __device__ __forceinline__ SymSlot(float hist_scale, int bins, bool clip, const int *sh)
        : cap((float)(clip ? bins : bins - 1)), base((uint32_t)__cvta_generic_to_shared(sh) - 0x4B000000u * 4u) { d.init(hist_scale); }
    __device__ __forceinline__ uint32_t addr(float q) const {
        return base + __float_as_uint(__fadd_rd(fminf(fmaxf(q, 0.f), cap), 8388608.f)) * 4u;
    }
    __device__ __forceinline__ static void count(uint32_t a) { asm volatile("red.shared.add.u32 [%0], 1;" ::"r"(a) : "memory"); }
    __device__ __forceinline__ void add(float v) const { count(addr(d.div(fabsf(v)))); }
    __device__ __forceinline__ void add4(const float4 &v) const {
        const float4 q = d.div4(make_float4(fabsf(v.x), fabsf(v.y), fabsf(v.z), fabsf(v.w)));
        count(addr(q.x)); count(addr(q.y)); count(addr(q.z)); count(addr(q.w));
    }
};

template <int TPB, int MINB, int U>
__global__ void __launch_bounds__(TPB, MINB)
multi_histogram_stream_kernel(const ppq_b200_tensor_desc *__restrict__ descs, int count, const float *__restrict__ hist_scale_arena,
                              int clip, int bins, int32_t *__restrict__ hist_arena) {
    extern __shared__ int sh[];
    int64_t *prefix = reinterpret_cast<int64_t *>(sh + ((bins + 1 + 1) & ~1));   // [count + 1], 8-byte aligned
    const int64_t total = build_prefix(descs, count, prefix);
    int64_t s0, s1; int t;
    if (!cta_span(prefix, count, total, s0, s1, t)) return;
    for (; t < count && prefix[t] < s1; t++) {
        const ppq_b200_tensor_desc d = descs[t];
        const int64_t a = max(s0 - prefix[t], (int64_t)0), b = min(s1 - prefix[t], d.n);
        if (b <= a) continue;                                          // uniform per CTA
        int32_t *gh = hist_arena + (int64_t)d.slot * bins;
        hist_zero<0>(sh, bins);
        const SymSlot bin(__ldg(hist_scale_arena + d.slot), bins, clip != 0, sh);
        stream_v8<U>(d.x + a, b - a, threadIdx.x, TPB, [&](const float4 &v) { bin.add4(v); }, [&](float v) { bin.add(v); });
        hist_flush<0>(sh, bins, gh);
    }
}

// ---- launch helpers -------------------------------------------------------------------------------------------------------
constexpr int kMaxSmemBins = 12287;            // (bins + 1) int32 slots within the default 48 KB of dynamic shared memory

// Elements each CTA should own before paying for zeroing + flushing `bins` counters.
static inline int hist_grid(int64_t n, int bins) {
    const int64_t per_cta = (int64_t)bins * 16 > 65536 ? (int64_t)bins * 16 : 65536;
    int64_t g = (n + per_cta - 1) / per_cta;
    const int64_t cap = (int64_t)sm_count();
    if (g > cap) g = cap;
    if (g < 1) g = 1;
    return (int)g;
}

template <class Bin>
static int launch_hist(const float *x, int64_t n, const BinParams &bin, int64_t bins, int32_t *hist, cudaStream_t st) {
    int var = variant_of(kVarHistogram);
    if (bins > kMaxSmemBins) var = 3;
    const int grid = var == 3 ? grid_for(n, kThreads, 16, 8) : hist_grid(n, (int)bins);
    const size_t smem = var == 3 ? 0 : (size_t)(bins + 1) * sizeof(int);
    switch (var) {
    case 1:  histogram_kernel<1, Bin><<<grid, kHistThreads, smem, st>>>(x, n, bin, hist); break;
    case 2:  histogram_kernel<2, Bin><<<grid, kHistThreads, smem, st>>>(x, n, bin, hist); break;
    case 3:  histogram_kernel<3, Bin, kUnroll, kThreads><<<grid, kThreads, smem, st>>>(x, n, bin, hist); break;
    case 4:  histogram_kernel<0, Bin, 8, kThreads><<<grid * 8 > sm_count() * 8 ? sm_count() * 8 : grid * 8, kThreads, smem, st>>>(x, n, bin, hist); break;   // the round-1 small-CTA layout
    // 5 / 6: two 1024-thread CTAs per SM (32 registers per thread), 2 / 4 loads in flight per thread
    case 5:  histogram_kernel<0, Bin><<<grid, kHistThreads, smem, st>>>(x, n, bin, hist); break;          // the round-1 default: one 1024-thread CTA per SM, 4 loads in flight
    case 6:  histogram_kernel<0, Bin, 4, kHistThreads, 2><<<grid * 2 > sm_count() * 2 ? sm_count() * 2 : grid * 2, kHistThreads, smem, st>>>(x, n, bin, hist); break;
    // 7 / 8: thread-block clusters of 2 / 4 CTAs, DSMEM pre-reduction of the private bins (grid rounded down to whole clusters)
    case 7:  if (grid >= 2) { histogram_cluster_kernel<Bin, 2><<<grid & ~1, kHistThreads, smem, st>>>(x, n, bin, hist); break; }
             histogram_kernel<0, Bin><<<grid, kHistThreads, smem, st>>>(x, n, bin, hist); break;
    case 8:  if (grid >= 4) { histogram_cluster_kernel<Bin, 4><<<grid & ~3, kHistThreads, smem, st>>>(x, n, bin, hist); break; }
             histogram_kernel<0, Bin><<<grid, kHistThreads, smem, st>>>(x, n, bin, hist); break;
    // default: two 1024-thread CTAs per SM (32 registers per thread), 2 loads in flight per thread
    default: histogram_kernel<0, Bin, 2, kHistThreads, 2><<<grid * 2 > sm_count() * 2 ? sm_count() * 2 : grid * 2, kHistThreads, smem, st>>>(x, n, bin, hist); break;
    }
    return (int)cudaGetLastError();
}

// Multi-tensor stream launches: one full wave of MINB CTAs per SM, each owning an equal span of the concatenation.  Both run 2 x 512
// threads per SM with 4 x 256-bit loads per thread in flight (128 KB per SM); measured on B200 against 512 x 4 (U 2), 1024 x 1 and,
// for the histogram, 1024 x 1 (U 2 / U 4) and 512 x 3 (U 2): profiles/r03_ab_explore.txt.
constexpr size_t kMaxPrefixSmem = 200 * 1024;  // descriptor prefix of the min/max launch: up to ~25 k tensors

template <int TPB, int MINB, int U>
static int launch_multi_minmax(const ppq_b200_tensor_desc *descs, int count, size_t smem, float *arena, cudaStream_t st) {
    auto k = multi_minmax_stream_kernel<TPB, MINB, U>;
    if (smem > 48 * 1024) {
        const cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return (int)e;
    }
    k<<<sm_count() * MINB, TPB, smem, st>>>(descs, count, arena);
    return (int)cudaGetLastError();
}

template <int TPB, int MINB, int U>
static int launch_multi_hist(const ppq_b200_tensor_desc *descs, int count, size_t smem, const float *hist_scale_arena, int clip,
                             int bins, int32_t *hist_arena, cudaStream_t st) {
    multi_histogram_stream_kernel<TPB, MINB, U><<<sm_count() * MINB, TPB, smem, st>>>(descs, count, hist_scale_arena, clip, bins, hist_arena);
    return (int)cudaGetLastError();
}

}  // namespace ppqb

using namespace ppqb;

extern "C" {

int ppq_b200_minmax_init(float *mins, float *maxs, int64_t count, void *stream) {
    if (count <= 0 || (!mins && !maxs)) return (int)cudaErrorInvalidValue;
    minmax_init_kernel<<<(int)((count + 255) / 256), 256, 0, (cudaStream_t)stream>>>(mins, maxs, count);
    return (int)cudaGetLastError();
}

int ppq_b200_minmax_t(const float *x, int64_t n, float *minmax, void *stream) {
    if (n <= 0 || !x || !minmax) return (int)cudaErrorInvalidValue;
    const int grid = grid_for((n + 3) / 4, kThreads, kUnroll * 4, 8);
    minmax_t_kernel<<<grid, kThreads, 0, (cudaStream_t)stream>>>(x, n, minmax);
    return (int)cudaGetLastError();
}

int ppq_b200_minmax_c(const float *x, int64_t n, int64_t epc, int C, float *mins, float *maxs, void *stream) {
    if (n <= 0 || epc <= 0 || C <= 0 || !x || !mins || !maxs || n % epc != 0) return (int)cudaErrorInvalidValue;
    const int64_t rows = n / epc;
    const int64_t chunks = (epc + kRowChunk - 1) / kRowChunk;
    if (chunks > 0x7fffffffLL) return (int)cudaErrorInvalidValue;
    const int64_t items = rows * chunks;
    int64_t grid = (items + (kThreads / 32) - 1) / (kThreads / 32);
    if (grid > (int64_t)sm_count() * 8) grid = (int64_t)sm_count() * 8;
    minmax_c_kernel<<<(int)grid, kThreads, 0, (cudaStream_t)stream>>>(x, rows, epc, C, chunks, FastDiv((uint32_t)chunks),
                                                                          FastDiv((uint32_t)C), mins, maxs);
    return (int)cudaGetLastError();
}

int ppq_b200_histogram_t(const float *x, int64_t n, float hist_scale, int clip_outliers, int32_t *hist, int64_t bins, void *stream) {
    if (n <= 0 || !x || !hist || bins <= 0 || bins > 0x7fffffffLL) return (int)cudaErrorInvalidValue;
    return launch_hist<SymBin>(x, n, BinParams{hist_scale, 0.f, (int)bins, clip_outliers}, bins, hist, (cudaStream_t)stream);
}

int ppq_b200_histogram_asym_t(const float *x, int64_t n, float vmin, float vmax, int clip_outliers, int32_t *hist, int64_t bins,
                              void *stream) {
    if (n <= 0 || !x || !hist || bins <= 0 || bins > 0x7fffffffLL) return (int)cudaErrorInvalidValue;
    return launch_hist<AsymBin>(x, n, BinParams{vmin, vmax, (int)bins, clip_outliers}, bins, hist, (cudaStream_t)stream);
}

int ppq_b200_histogram_t_dscale(const float *x, int64_t n, const float *hist_scale_dev, int clip_outliers, int32_t *hist,
                                int64_t bins, void *stream) {
    if (n <= 0 || !x || !hist || !hist_scale_dev || bins <= 0 || bins > kMaxSmemBins) return (int)cudaErrorInvalidValue;
    const int grid = hist_grid(n, (int)bins) * 2 > sm_count() * 2 ? sm_count() * 2 : hist_grid(n, (int)bins) * 2;
    histogram_dscale_kernel<0><<<grid, kHistThreads, (size_t)(bins + 1) * sizeof(int), (cudaStream_t)stream>>>(
        x, n, hist_scale_dev, clip_outliers, (int)bins, hist);
    return (int)cudaGetLastError();
}

int ppq_b200_histogram_c(const float *x, int64_t n, int64_t epc, int C, float hist_scale, int clip_outliers, int32_t *hist,
                         int64_t bins, void *stream) {
    if (n <= 0 || epc <= 0 || C <= 0 || !x || !hist || bins <= 0 || bins > kMaxSmemBins || n % epc != 0)
        return (int)cudaErrorInvalidValue;
    const int64_t rows = n / epc;
    const int64_t chunk = (int64_t)bins * 8 > 32768 ? (int64_t)bins * 8 : 32768;
    const int64_t chunks = (epc + chunk - 1) / chunk;
    const int64_t items = rows * chunks;
    const int grid = (int)(items < (int64_t)sm_count() * 8 ? items : (int64_t)sm_count() * 8);
    histogram_c_kernel<0><<<grid, kThreads, (size_t)(bins + 1) * sizeof(int), (cudaStream_t)stream>>>(
        x, rows, epc, C, chunk, chunks, hist_scale, clip_outliers, (int)bins, hist);
    return (int)cudaGetLastError();
}

int ppq_b200_multi_minmax_t(const ppq_b200_tensor_desc *descs, int count, int64_t max_n, float *minmax_arena, void *stream) {
    if (count <= 0 || max_n <= 0 || !descs || !minmax_arena) return (int)cudaErrorInvalidValue;
    if (variant_of(kVarMinMax) != 1) {          // 1: the replaced per-chunk kernel below (A/B only)
        const size_t smem = (size_t)(count + 1) * sizeof(int64_t);
        if (smem > kMaxPrefixSmem) return (int)cudaErrorInvalidValue;
        return launch_multi_minmax<512, 2, 4>(descs, count, smem, minmax_arena, (cudaStream_t)stream);
    }
    const int64_t chunk = 65536;
    const int64_t cpt = (max_n + chunk - 1) / chunk;
    if (cpt > 0x7fffffffLL) return (int)cudaErrorInvalidValue;
    const int64_t items = (int64_t)count * cpt;
    const int grid = (int)(items < (int64_t)sm_count() * 8 ? items : (int64_t)sm_count() * 8);
    multi_minmax_t_kernel<<<grid, kThreads, 0, (cudaStream_t)stream>>>(descs, count, chunk, (int)cpt, minmax_arena);
    return (int)cudaGetLastError();
}

int ppq_b200_multi_histogram_t(const ppq_b200_tensor_desc *descs, int count, int64_t max_n, const float *hist_scale_arena,
                               int clip_outliers, int32_t *hist_arena, int64_t bins, void *stream) {
    if (count <= 0 || max_n <= 0 || !descs || !hist_scale_arena || !hist_arena || bins <= 0 || bins > kMaxSmemBins) return (int)cudaErrorInvalidValue;
    const size_t smem = (size_t)((bins + 2) & ~1) * sizeof(int) + (size_t)(count + 1) * sizeof(int64_t);
    if (smem > 48 * 1024) return (int)cudaErrorInvalidValue;
    if (variant_of(kVarMultiHist) != 1) {       // 1: the replaced fixed-span kernel below (A/B only)
        return launch_multi_hist<512, 2, 4>(descs, count, smem, hist_scale_arena, clip_outliers, (int)bins, hist_arena, (cudaStream_t)stream);
    }
    // grid: one CTA per SM, fewer when the whole job is small (each CTA should own >= 64 Ki elements before paying for a flush)
    int64_t g = ((int64_t)count * max_n + 65535) / 65536;
    if (g > sm_count()) g = sm_count();
    if (g < 1) g = 1;
    multi_histogram_t_kernel<0><<<(int)g, kHistThreads, smem, (cudaStream_t)stream>>>(descs, count, hist_scale_arena, clip_outliers, (int)bins,
                                                                                      hist_arena);
    return (int)cudaGetLastError();
}

}  // extern "C"
