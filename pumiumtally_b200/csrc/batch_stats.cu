// Batch statistics kernels (Engine::end_batch, get_tally_statistics, max_relative_error): the running
// sums S1 = sum of batch values and S2 = sum of their squares per (bin, element), and what is read out of
// them.  The per-element arithmetic is in batch_stats.cuh.
//
// The accumulate pass runs between two moves.  Its four streams (batch value, zero written back, S1, S2:
// 48 bytes per entry) are touched once each, so they are loaded and stored with L1::no_allocate and an
// L2 evict_first policy, the way the walk streams particle data: the tet records the walk keeps with
// evict_last (on config c2 the 128 MB table only half-fits the 126 MB L2) are what the next move needs.
#include <climits>
#include <cstdint>

#include "batch_stats.cuh"

namespace ptb {
namespace {

constexpr int kBlock = 256;

__device__ __forceinline__ unsigned long long evict_first_policy() {
  unsigned long long p;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
  return p;
}

struct D4 { double a, b, c, d; };

__device__ __forceinline__ D4 load4(const double *p, unsigned long long pol) {
  D4 v;
  asm volatile("ld.global.L1::no_allocate.L2::cache_hint.v4.f64 {%0,%1,%2,%3}, [%4], %5;"
               : "=d"(v.a), "=d"(v.b), "=d"(v.c), "=d"(v.d) : "l"(p), "l"(pol));
  return v;
}

__device__ __forceinline__ void store4(double *p, const D4 &v, unsigned long long pol) {
  asm volatile("st.global.L1::no_allocate.L2::cache_hint.v4.f64 [%0], {%1,%2,%3,%4}, %5;"
               ::"l"(p), "d"(v.a), "d"(v.b), "d"(v.c), "d"(v.d), "l"(pol) : "memory");
}

__device__ __forceinline__ double load1(const double *p, unsigned long long pol) {
  double v;
  asm volatile("ld.global.L1::no_allocate.L2::cache_hint.f64 %0, [%1], %2;" : "=d"(v) : "l"(p), "l"(pol));
  return v;
}

__device__ __forceinline__ void store1(double *p, double v, unsigned long long pol) {
  asm volatile("st.global.L1::no_allocate.L2::cache_hint.f64 [%0], %1, %2;" ::"l"(p), "d"(v), "l"(pol) : "memory");
}

// vec4: x, zero_out, s1 and s2 are 32-byte aligned, so groups of four entries move as 256-bit accesses
__global__ void batch_accumulate_kernel(const double *x, double divisor, double *zero_out, double *s1, double *s2,
                                        int64_t count, bool first, bool vec4) {
  const unsigned long long pol = evict_first_policy();
  const int64_t stride = (int64_t)gridDim.x * blockDim.x, tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  int64_t done = 0;
  if (vec4) {
    const int64_t groups = count / 4;
    for (int64_t g = tid; g < groups; g += stride) {
      const int64_t j = 4 * g;
      const D4 v = load4(x + j, pol);
      D4 a = load4(s1 + j, pol), b = load4(s2 + j, pol);
      batch_accumulate(v.a / divisor, a.a, b.a, first);
      batch_accumulate(v.b / divisor, a.b, b.b, first);
      batch_accumulate(v.c / divisor, a.c, b.c, first);
      batch_accumulate(v.d / divisor, a.d, b.d, first);
      store4(s1 + j, a, pol);
      store4(s2 + j, b, pol);
      if (zero_out) store4(zero_out + j, D4{0.0, 0.0, 0.0, 0.0}, pol);
    }
    done = 4 * groups;
  }
  for (int64_t j = done + tid; j < count; j += stride) {
    double a = load1(s1 + j, pol), b = load1(s2 + j, pol);
    batch_accumulate(load1(x + j, pol) / divisor, a, b, first);
    store1(s1 + j, a, pol);
    store1(s2 + j, b, pol);
    if (zero_out) store1(zero_out + j, 0.0, pol);
  }
}

__global__ void batch_finish_kernel(const double *s1, const double *s2, int64_t count, int64_t offset, int64_t E,
                                    const double *volume, double n, double *mean, double *std_dev) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; j < count; j += stride) {
    const double vol = __ldg(volume + (offset + j) % E), a = s1[j];
    mean[j] = batch_mean(a, n, vol);
    std_dev[j] = batch_std_dev(a, s2[j], n, vol);
  }
}

// (rel, idx) ordering of the trigger: larger relative error first, then the lower index
__device__ __forceinline__ bool better(double r, long long i, double r0, long long i0) {
  return r > r0 || (r == r0 && i < i0);
}

// block-wide reduction of (rel, idx, cnt); thread 0 gets the result
__device__ void block_reduce(double &rel, long long &idx, unsigned long long &cnt) {
  __shared__ double s_rel[kBlock / 32];
  __shared__ long long s_idx[kBlock / 32];
  __shared__ unsigned long long s_cnt[kBlock / 32];
  for (int d = 16; d > 0; d >>= 1) {
    const double r = __shfl_down_sync(0xffffffffu, rel, d);
    const long long i = __shfl_down_sync(0xffffffffu, idx, d);
    cnt += __shfl_down_sync(0xffffffffu, cnt, d);
    if (better(r, i, rel, idx)) { rel = r; idx = i; }
  }
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (lane == 0) { s_rel[warp] = rel; s_idx[warp] = idx; s_cnt[warp] = cnt; }
  __syncthreads();
  if (warp == 0) {
    const bool have = lane < kBlock / 32;
    rel = have ? s_rel[lane] : -1.0;
    idx = have ? s_idx[lane] : LLONG_MAX;
    cnt = have ? s_cnt[lane] : 0ull;
    for (int d = 16; d > 0; d >>= 1) {
      const double r = __shfl_down_sync(0xffffffffu, rel, d);
      const long long i = __shfl_down_sync(0xffffffffu, idx, d);
      cnt += __shfl_down_sync(0xffffffffu, cnt, d);
      if (better(r, i, rel, idx)) { rel = r; idx = i; }
    }
  }
}

__global__ void __launch_bounds__(kBlock) batch_trigger_kernel(const double *s1, const double *s2, int64_t count,
                                                               int64_t offset, int64_t E, const double *volume,
                                                               const int32_t *orig_of_internal, double n,
                                                               double threshold, double *partial) {
  double best = -1.0;
  long long best_idx = LLONG_MAX;
  unsigned long long above = 0;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; j < count; j += stride) {
    const int64_t g = offset + j, bin = g / E, elem = g - bin * E;
    const double vol = __ldg(volume + elem), a = s1[j];
    const double rel = batch_relative_error(batch_mean(a, n, vol), batch_std_dev(a, s2[j], n, vol));
    if (rel < 0.0) continue;  // zero mean (a NaN ratio fails every comparison below as well)
    if (rel > threshold) ++above;
    const long long idx = bin * E + __ldg(orig_of_internal + elem);
    if (better(rel, idx, best, best_idx)) { best = rel; best_idx = idx; }
  }
  block_reduce(best, best_idx, above);
  if (threadIdx.x == 0) {
    partial[3 * blockIdx.x] = best;
    partial[3 * blockIdx.x + 1] = best < 0.0 ? -1.0 : double(best_idx);
    partial[3 * blockIdx.x + 2] = double(above);
  }
}

// one block: the per-block records -> out[3]
__global__ void __launch_bounds__(kBlock) batch_trigger_final_kernel(const double *partial, int nparts, double *out) {
  double best = -1.0;
  long long best_idx = LLONG_MAX;
  unsigned long long above = 0;
  for (int k = threadIdx.x; k < nparts; k += blockDim.x) {
    above += (unsigned long long)partial[3 * k + 2];
    const double r = partial[3 * k];
    const long long i = partial[3 * k + 1] < 0.0 ? LLONG_MAX : (long long)partial[3 * k + 1];
    if (r >= 0.0 && better(r, i, best, best_idx)) { best = r; best_idx = i; }
  }
  block_reduce(best, best_idx, above);
  if (threadIdx.x == 0) {
    out[0] = best;
    out[1] = best < 0.0 ? -1.0 : double(best_idx);
    out[2] = double(above);
  }
}

int grid_for(int64_t items, int max_blocks) {
  const int64_t b = (items + kBlock - 1) / kBlock;
  return int(b < 1 ? 1 : (b > max_blocks ? max_blocks : b));
}

bool aligned32(const void *p) { return (reinterpret_cast<uintptr_t>(p) & 31u) == 0; }

}  // namespace

cudaError_t launch_batch_accumulate(const double *x, double divisor, double *zero_out, double *s1, double *s2,
                                    int64_t count, bool first, cudaStream_t stream) {
  if (count <= 0) return cudaSuccess;
  const bool vec4 = aligned32(x) && aligned32(zero_out) && aligned32(s1) && aligned32(s2);
  batch_accumulate_kernel<<<grid_for(vec4 ? (count + 3) / 4 : count, 148 * 8), kBlock, 0, stream>>>(
      x, divisor, zero_out, s1, s2, count, first, vec4);
  return cudaGetLastError();
}

cudaError_t launch_batch_finish(const double *s1, const double *s2, int64_t count, int64_t offset, int64_t E,
                                const double *volume, double n, double *mean, double *std_dev, cudaStream_t stream) {
  if (count <= 0) return cudaSuccess;
  batch_finish_kernel<<<grid_for(count, 148 * 8), kBlock, 0, stream>>>(s1, s2, count, offset, E, volume, n, mean, std_dev);
  return cudaGetLastError();
}

cudaError_t launch_batch_trigger(const double *s1, const double *s2, int64_t count, int64_t offset, int64_t E,
                                 const double *volume, const int32_t *orig_of_internal, double n, double threshold,
                                 double *partial, double *out, cudaStream_t stream) {
  const int blocks = grid_for(count, kBatchTriggerBlocks);
  batch_trigger_kernel<<<blocks, kBlock, 0, stream>>>(s1, s2, count < 0 ? 0 : count, offset, E, volume,
                                                      orig_of_internal, n, threshold, partial);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return e;
  batch_trigger_final_kernel<<<1, kBlock, 0, stream>>>(partial, blocks, out);
  return cudaGetLastError();
}

}  // namespace ptb
