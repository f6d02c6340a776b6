#!/usr/bin/env python
"""HBM read ceiling of this GPU: how fast a read-only stream (a trivial reduction) and a device-to-device copy go.

    python tools/hbm_ceiling.py [--gb 2.7] [--buffers 4] [--reps 3] [--out FILE]

The collectors (multi_minmax_t, multi_histogram_t) only read, so their share of peak is taken against the read ceiling; the copy ceiling
(MEASURED_PEAKS.json hbm_gbs, read + write) is measured in the same run for comparison.  Its own kernels are compiled with nvcc into a
temporary directory.  Each pass reads one of `buffers` rotating buffers of `gb` GB, so no pass finds its data in the 126 MB L2.
Sweeps 128- vs 256-bit loads, 4 vs 8 loads in flight per thread, three CTA sizes (grid = one full wave at the occupancy the compiler
allows) and the L2::256B prefetch hint (with L2::evict_first on the 256-bit loads; the 128-bit
form does not take it).
"""
import argparse
import ctypes
import os
import subprocess
import sys
import tempfile

import torch

SRC = r'''
#include <cuda_runtime.h>
#include <stdint.h>

template <int BYTES, bool HINT> struct Ld;
template <> struct Ld<16, false> { static __device__ __forceinline__ float sum(const float *p) { float a, b, c, d;
    asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(a), "=f"(b), "=f"(c), "=f"(d) : "l"(p)); return (a + b) + (c + d); } };
template <> struct Ld<16, true> { static __device__ __forceinline__ float sum(const float *p) { float a, b, c, d;
    asm volatile("ld.global.nc.L1::no_allocate.L2::256B.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(a), "=f"(b), "=f"(c), "=f"(d) : "l"(p)); return (a + b) + (c + d); } };
template <> struct Ld<32, false> { static __device__ __forceinline__ float sum(const float *p) { float a, b, c, d, e, f, g, h;
    asm volatile("ld.global.nc.L1::no_allocate.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=f"(a), "=f"(b), "=f"(c), "=f"(d), "=f"(e), "=f"(f), "=f"(g), "=f"(h) : "l"(p)); return ((a + b) + (c + d)) + ((e + f) + (g + h)); } };
template <> struct Ld<32, true> { static __device__ __forceinline__ float sum(const float *p) { float a, b, c, d, e, f, g, h;
    asm volatile("ld.global.nc.L1::no_allocate.L2::evict_first.L2::256B.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=f"(a), "=f"(b), "=f"(c), "=f"(d), "=f"(e), "=f"(f), "=f"(g), "=f"(h) : "l"(p)); return ((a + b) + (c + d)) + ((e + f) + (g + h)); } };

// Sum of n floats (n a multiple of the segment), lane-interleaved vectors in warp-contiguous segments of 32 x U vectors.
template <int BYTES, int U, bool HINT>
__global__ void read_kernel(const float *__restrict__ x, int64_t n, float *out) {
    constexpr int F = BYTES / 4, SEG = 32 * F * U;
    const int64_t warps = (int64_t)gridDim.x * blockDim.x / 32;
    float acc = 0.f;
    for (int64_t s = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) / 32 * SEG + (threadIdx.x & 31) * F; s < n; s += warps * SEG) {
        float v[U];
#pragma unroll
        for (int j = 0; j < U; j++) v[j] = Ld<BYTES, HINT>::sum(x + s + j * 32 * F);
#pragma unroll
        for (int j = 0; j < U; j++) acc += v[j];
    }
    if (acc == 123.456f) out[0] = acc;                                  // keeps the sum alive
}

__global__ void copy_kernel(const float4 *__restrict__ x, float4 *__restrict__ y, int64_t n4) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) y[i] = x[i];
}

template <class K> static int wave(K k, int threads) {
    int dev = 0, sms = 0, per = 0;
    cudaGetDevice(&dev); cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per, k, threads, 0);
    return sms * (per > 0 ? per : 1);
}

extern "C" int read_stream(int bytes, int unroll, int hint, int threads, const float *x, int64_t n, float *out, int *grid) {
#define CASE(B, U, H) if (bytes == B && unroll == U && hint == H) { auto k = read_kernel<B, U, H>; *grid = wave(k, threads); \
        k<<<*grid, threads>>>(x, n, out); return (int)cudaGetLastError(); }
    CASE(16, 4, false) CASE(16, 8, false) CASE(16, 4, true) CASE(16, 8, true)
    CASE(32, 4, false) CASE(32, 8, false) CASE(32, 4, true) CASE(32, 8, true)
    return -1;
}
extern "C" int copy_stream(const float *x, float *y, int64_t n, int threads, int *grid) {
    *grid = wave(copy_kernel, threads);
    copy_kernel<<<*grid, threads>>>(reinterpret_cast<const float4 *>(x), reinterpret_cast<float4 *>(y), n / 4);
    return (int)cudaGetLastError();
}
'''


def compile_lib(tmp):
    src = os.path.join(tmp, 'hbm_ceiling.cu')
    lib = os.path.join(tmp, 'libhbm_ceiling.so')
    open(src, 'w').write(SRC)
    nvcc = os.environ.get('NVCC', '/usr/local/cuda/bin/nvcc')
    subprocess.run([nvcc, '-gencode', 'arch=compute_100a,code=sm_100a', '-O3', '-std=c++17', '-shared', '-Xcompiler', '-fPIC',
                    src, '-o', lib], check=True)
    return ctypes.CDLL(lib)


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(['nvidia-smi', '-i', '0', '--query-gpu=power.limit,clocks.sm,clocks.max.sm,clocks.mem', '--format=csv,noheader'],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:                                                # noqa: BLE001
        q = f'nvidia-smi unavailable ({type(e).__name__})'
    return f'{name}; power limit, SM clock, max SM clock, memory clock: {q}'


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gb', type=float, default=2.7)
    ap.add_argument('--buffers', type=int, default=4)
    ap.add_argument('--reps', type=int, default=3, help='passes over every buffer per configuration')
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), 'the probe measures a GPU'
    lines = []

    def say(s):
        print(s, flush=True); lines.append(s)
    with tempfile.TemporaryDirectory() as tmp:
        lib = compile_lib(tmp)
        seg = 32 * 8 * 8
        n = int(args.gb * 1e9 / 4) // seg * seg
        bufs = [torch.ones(n, device='cuda') for _ in range(args.buffers)]
        dst = torch.empty(n, device='cuda')
        out = torch.zeros(1, device='cuda')
        grid = ctypes.c_int(0)
        say(card())
        say(f'{args.buffers} rotating buffers of {4 * n / 1e9:.3f} GB, {args.reps} passes over each per configuration; CUDA events')

        def timed(launch):
            for b in bufs[:2]: launch(b)                                 # warm-up
            a, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize(); a.record()
            for _ in range(args.reps):
                for b in bufs: launch(b)
            e.record(); torch.cuda.synchronize()
            return a.elapsed_time(e) * 1e-3 / (args.reps * len(bufs))

        best = (0.0, '')
        for threads in (256, 512, 1024):
            for bytes_ in (16, 32):
                for unroll in (4, 8):
                    for hint in (0, 1):
                        def launch(b):
                            rc = lib.read_stream(bytes_, unroll, hint, threads, ctypes.c_void_p(b.data_ptr()), ctypes.c_int64(n),
                                                 ctypes.c_void_p(out.data_ptr()), ctypes.byref(grid))
                            assert rc == 0, rc
                        s = timed(launch)
                        gbs = 4 * n / s / 1e9
                        cfg = f'read  {8 * bytes_:3d}-bit x {unroll} in flight, {threads:4d} thr x {grid.value // torch.cuda.get_device_properties(0).multi_processor_count} CTA/SM, hints {"on " if hint else "off"}'
                        say(f'{cfg}: {s * 1e3:7.4f} ms  {gbs:7.1f} GB/s')
                        if gbs > best[0]: best = (gbs, cfg)
        for threads in (256, 1024):
            def launch(b):
                assert lib.copy_stream(ctypes.c_void_p(b.data_ptr()), ctypes.c_void_p(dst.data_ptr()), ctypes.c_int64(n), threads, ctypes.byref(grid)) == 0
            s = timed(launch)
            say(f'copy  128-bit, {threads:4d} thr, grid {grid.value}: {s * 1e3:7.4f} ms  {8 * n / s / 1e9:7.1f} GB/s (read + write)')
        say(f'read ceiling: {best[0]:.1f} GB/s ({best[1]})')
    if args.out:
        with open(args.out, 'w') as f: f.write('\n'.join(lines) + '\n')


if __name__ == '__main__':
    sys.exit(main())
