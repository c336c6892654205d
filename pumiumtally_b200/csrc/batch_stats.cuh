// Per-element arithmetic of the batch statistics (batch_stats.cu, Engine::end_batch): running sums of the
// batch values and of their squares, and from them the mean and the standard deviation of the mean
// (OpenMC's tally statistics).
//
// The functions are __host__ __device__ only so that tests/ can compile them with g++ and check them
// against numpy on a machine without a GPU; the library runs them on the device only.  Every
// multiply-add is written as an explicit fma so that the host build, the finish kernel and the trigger
// kernel round identically (nvcc would otherwise be free to contract some of them and not others).
#pragma once
#include <cstdint>

#if defined(__CUDACC__)
#define PTB_BS_HD __host__ __device__ __forceinline__
#else
#define PTB_BS_HD inline
#endif
#include <cmath>

namespace ptb {

// s1 += x, s2 += x^2; `first` starts the sums over (the accumulators need no clearing after a reset)
PTB_BS_HD void batch_accumulate(double x, double &s1, double &s2, bool first) {
  s1 = (first ? 0.0 : s1) + x;
  s2 = fma(x, x, first ? 0.0 : s2);
}

// mean of n batch values per unit volume: S1 / n / volume
PTB_BS_HD double batch_mean(double s1, double n, double volume) { return s1 / n / volume; }

// Standard deviation of the mean per unit volume: sqrt((S2/n - (S1/n)^2) / (n - 1)) / volume.  A negative
// rounding residue of the variance (identical batches) is clamped to 0; with fewer than two batches the
// result is NaN.
PTB_BS_HD double batch_std_dev(double s1, double s2, double n, double volume) {
  if (!(n >= 2.0)) return NAN;
  const double m = s1 / n, q = s2 / n;
  const double var = fma(-m, m, q) / (n - 1.0);
  return sqrt(var > 0.0 ? var : 0.0) / volume;
}

// one (bin, element) pair's contribution to the relative-error trigger: std_dev / |mean|, or -1 when the
// mean is zero (such pairs are left out)
PTB_BS_HD double batch_relative_error(double mean, double std_dev) {
  return mean != 0.0 ? std_dev / fabs(mean) : -1.0;
}

}  // namespace ptb

#if defined(__CUDACC__)
#include <cuda_runtime.h>

namespace ptb {

// Launch interface of batch_stats.cu.  Every pass covers one rank's share of the bin-major tally: entries
// j in [0, count), whose bin-major index is offset + j (element (offset + j) % E of bin (offset + j) / E).
//
// With v = x[j] / divisor (the batch value): S1[j], S2[j] += v, v^2 (first: S1, S2 = v, v^2); zero_out (may be
// null, may equal x) gets a 0.0 in every slot read.  All four arrays are streamed with L2::evict_first.
cudaError_t launch_batch_accumulate(const double *x, double divisor, double *zero_out, double *s1, double *s2,
                                    int64_t count, bool first, cudaStream_t stream);
// mean[j], std_dev[j] of n batches, per unit volume
cudaError_t launch_batch_finish(const double *s1, const double *s2, int64_t count, int64_t offset, int64_t E,
                                const double *volume, double n, double *mean, double *std_dev, cudaStream_t stream);
// Trigger query over the share: out[0] = largest std_dev / |mean| over entries with mean != 0 (-1 if there
// is none), out[1] = bin * E + orig_of_internal[element] where it is reached (lowest such index on ties),
// out[2] = number of entries whose relative error exceeds `threshold`.  partial: room for
// kBatchTriggerBlocks records of 3 doubles.
constexpr int kBatchTriggerBlocks = 592;
cudaError_t launch_batch_trigger(const double *s1, const double *s2, int64_t count, int64_t offset, int64_t E,
                                 const double *volume, const int32_t *orig_of_internal, double n, double threshold,
                                 double *partial, double *out, cudaStream_t stream);

}  // namespace ptb
#endif
