// Ordered scatter-reduce for Reduction.sum / mean / prod (utils.py:70-76).
//
// torch_scatter's CPU kernels (and ATen's scatter_reduce_, which the fixtures were generated with) walk the points
// of a row in index order and fold each into its cell: out[idx[i]] = out[idx[i]] (+|*) src[i].  Floating-point sums
// and products depend on that order, so an atomicAdd scatter agrees with the reference only to rounding, differently
// on every run, and the "cell changed" mask (utils.py:489-491: new != old) can flip where a sum lands exactly on the
// fill value.  Here the order is reproduced instead: every point gets the key (cell of the output), a STABLE radix
// sort (cub::DeviceRadixSort) brings the hits of a cell together in ascending point index, and one thread per cell
// folds them in that order with the reference's single-rounding operations.  Result: bit-identical to the CPU
// reference and deterministic.  max / min never come here (they are order-independent atomics in the other kernels).
#include <cub/device/device_radix_sort.cuh>

#include "dm_common.cuh"

namespace dm {

constexpr int kOrdThreads = 256;
constexpr unsigned long long kNoCell = ~0ull;

static unsigned ord_grid(long long items) {
  long long blocks = (items + kOrdThreads - 1) / kOrdThreads;
  const long long cap = (long long)sm_count() * 8 * 4;
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  return (unsigned)blocks;
}

// One thread per segment head: folds the segment's values, in sorted (= point index) order, into the cell.
// `values` is indexed by the payload.  reduction: 2 sum, 3 mean, 4 prod.
// mask_or (optional): the cell's "changed" flag of utils.py:489-491 — |new - old| with NaN counted as 0 — is set
// where it is true (cells nobody hits keep what the mask held).
__global__ void __launch_bounds__(kOrdThreads)
ordered_fold_kernel(const unsigned long long* __restrict__ keys, const unsigned int* __restrict__ payload,
                    const float* __restrict__ values, long long n, int reduction, float* __restrict__ canvas,
                    uint8_t* __restrict__ mask_or) {
  for (long long p = (long long)blockIdx.x * kOrdThreads + threadIdx.x; p < n; p += (long long)gridDim.x * kOrdThreads) {
    const unsigned long long k = keys[p];
    if (k == kNoCell) continue;
    if (p > 0 && keys[p - 1] == k) continue;  // not the first hit of its cell
    float acc = canvas[k];                    // the filled (or caller-provided) canvas takes part (utils.py:472-477)
    long long hits = 0;
    for (long long q = p; q < n && keys[q] == k; ++q) {
      const float v = values[payload[q]];
      acc = reduction == 4 ? __fmul_rn(acc, v) : __fadd_rn(acc, v);
      ++hits;
    }
    // scatter_mean: the sum (canvas included) divided by the number of hits (canvas excluded), at least 1.
    // torch_scatter counts with float32 ones, so its count stops at 2^24 (2^24 + 1 rounds back to 2^24).
    if (reduction == 3) acc = __fdiv_rn(acc, hits < (1ll << 24) ? (float)hits : 16777216.0f);
    if (mask_or) {
      float dlt = fabsf(__fsub_rn(acc, canvas[k]));
      if (dlt != dlt) dlt = 0.0f;
      if (dlt != 0.0f) mask_or[k] = 1;
    }
    canvas[k] = acc;
  }
}

__global__ void __launch_bounds__(kOrdThreads) iota_kernel(unsigned int* p, long long n) {
  for (long long i = (long long)blockIdx.x * kOrdThreads + threadIdx.x; i < n; i += (long long)gridDim.x * kOrdThreads)
    p[i] = (unsigned int)i;
}

// keys (n, device, consumed), values (indexed by point index), canvas holding the starting values.
// n < 2^31.  key_bits: number of significant key bits (the sentinel kNoCell has all bits set: it sorts last whatever
// the bit range, because every real key is smaller in the examined bits only if key_bits covers them; the sentinel's
// examined bits are all ones, so real keys must stay below 2^key_bits - 1).
int ordered_reduce(unsigned long long* keys, const float* values, long long n, int key_bits, int reduction,
                   float* canvas, uint8_t* mask_or, cudaStream_t stream) {
  if (n <= 0) return DM_OK;
  if (n >= (1ll << 31) || reduction < 2 || reduction > 4) return DM_EINVAL;
  unsigned long long* keys_out = nullptr;
  unsigned int *pay_in = nullptr, *pay_out = nullptr;
  void* temp = nullptr;
  size_t temp_bytes = 0;
  int end_bit = key_bits + 1;
  if (end_bit > 64) end_bit = 64;
  DM_CUDA_OK(cub::DeviceRadixSort::SortPairs(nullptr, temp_bytes, keys, keys_out, pay_in, pay_out, (int)n, 0, end_bit,
                                             stream));
  DM_CUDA_OK(cudaMallocAsync(&keys_out, (size_t)n * 8, stream));
  DM_CUDA_OK(cudaMallocAsync(&pay_in, (size_t)n * 4, stream));
  DM_CUDA_OK(cudaMallocAsync(&pay_out, (size_t)n * 4, stream));
  DM_CUDA_OK(cudaMallocAsync(&temp, temp_bytes ? temp_bytes : 16, stream));
  iota_kernel<<<ord_grid(n), kOrdThreads, 0, stream>>>(pay_in, n);
  DM_LAUNCHED();
  DM_CUDA_OK(cub::DeviceRadixSort::SortPairs(temp, temp_bytes, keys, keys_out, pay_in, pay_out, (int)n, 0, end_bit,
                                             stream));
  ++g_launches;
  ordered_fold_kernel<<<ord_grid(n), kOrdThreads, 0, stream>>>(keys_out, pay_out, values, n, reduction, canvas, mask_or);
  DM_LAUNCHED();
  DM_CUDA_OK(cudaFreeAsync(keys_out, stream));
  DM_CUDA_OK(cudaFreeAsync(pay_in, stream));
  DM_CUDA_OK(cudaFreeAsync(pay_out, stream));
  DM_CUDA_OK(cudaFreeAsync(temp, stream));
  return DM_OK;
}

int bits_for(unsigned long long max_key_exclusive) {  // smallest k with max_key_exclusive <= 2^k - 1
  int k = 1;
  while (k < 63 && ((1ull << k) - 1ull) < max_key_exclusive) ++k;
  return k;
}

}  // namespace dm
