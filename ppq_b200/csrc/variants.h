// variants.h -- run-time kernel variant selection (profiling / A-B benchmarking knob, see ppq_b200_set_variant).
//   "linear_quant_t": 0 default (LDG.128, warp-contiguous segments, unroll by size) | 1 TMA-staged smem ring | 2 force 8 loads in flight
//                     | 3 force 4 loads in flight on a persistent 148 x 8 grid
//   "histogram":      0 default (two 1024-thr CTAs per SM, 2 loads in flight, unconditional red.shared + trash slot) | 1 generic-pointer atomicAdd
//                     | 2 __match_any_sync aggregation | 3 global atomics like the reference | 4 the first layout (256-thr CTAs x 8 per SM)
//                     | 5 the round-1 default (one 1024-thr CTA per SM, 4 loads in flight) | 6 two CTAs per SM, 4 loads in flight | 7, 8 clusters of 2 / 4 CTAs, DSMEM pre-reduction of the bins
//   "minmax":         multi-tensor min/max: 0 default (equal spans of the concatenated tensors, 2 x 512-thr CTAs per SM, 4 x 256-bit loads in
//                     flight, per-warp publish) | 1 the replaced kernel (fixed 64 Ki-element chunks per tensor, empty items for small tensors)
//   "multi_histogram": 0 default (same spans and loads, full-rate floor into the shared-memory slot address) | 1 the replaced kernel
//                     (one 1024-thr CTA per SM, 128-bit loads, F2I per element)
//   "linear_quant_c": 0 default (shared-memory operator table for rows shorter than 512 elements) | 1 the round-1 per-vector operator rebuild
//   "kl_search": 0 default (one warp per candidate) | 1 the serial-candidate kernel
//   "select": single-tensor radix select A/B: low 3 bits = pass 0 (0 default: 2 x 1024 threads per SM, 4 interleaved loads | 1 two loads | 2 warp segments, 4 loads
//             | 3 warp segments, 2 loads | 4 four 512-thread CTAs), bits 3-5 = pass 1 (0 default: 6 x 256 threads, warp segments, 4 loads | 1 two loads | 2 3 x 512 threads | 3 2 x 1024 threads, 2 loads | 4 interleaved), bit 6 (64) = no thresholds from a sample on cold calls
#pragma once
namespace ppqb {
enum { kVarLinearT = 0, kVarHistogram = 1, kVarMinMax = 2, kVarChannel = 3, kVarKlSearch = 4, kVarSelect = 5, kVarMultiHist = 6, kVarCount = 8 };
int variant_of(int key);
}
