// Per-move spatial binning of the flying particles (counting sort by the Morton rank of the
// seed-grid cell of the particle's origin).  Output: order[] = ids of the flying
// particles of the range grouped by cell, and the number of them.  The walk
// kernel then processes particles in that order, so the lanes of a warp, the
// warps of a block and the blocks in flight at any moment work on neighbouring
// tets: tet records are served from L1/L2 instead of HBM.
//
// The reference has no counterpart (it re-streams every particle slot every
// iteration in storage order, SURVEY.md section 2b); results do not depend on
// the processing order except for the fp64 summation order of the atomics.
#include <cstdint>

#include "walk_kernels.hpp"

namespace ptb {
namespace {

constexpr int kScanBlock = 1024;  // elements per scan block (256 threads x 4)

__device__ __forceinline__ int32_t cell_of(const SeedGrid &g, double x, double y, double z) {
  // clamp into the grid: origins outside the bounding box land in the nearest cell
  const double fx = (x - g.x0) * g.inv_h, fy = (y - g.y0) * g.inv_h, fz = (z - g.z0) * g.inv_h;
  const int cx = fx > 0.0 ? min((int)fx, g.nx - 1) : 0;
  const int cy = fy > 0.0 ? min((int)fy, g.ny - 1) : 0;
  const int cz = fz > 0.0 ? min((int)fz, g.nz - 1) : 0;
  const int32_t c = (cz * g.ny + cy) * g.nx + cx;
  return g.cell_rank ? __ldg(g.cell_rank + c) : c;  // Morton rank of the cell = the bin
}

// pass 1: cell of every flying particle of [begin,end) + histogram
// origin == nullptr: every particle starts this move where it is; the key is then the stored position
__global__ void bin_count_kernel(SeedGrid g, const double *__restrict__ origin, const ParticleState *__restrict__ state,
                                 const int8_t *__restrict__ flying, int32_t begin, int32_t end,
                                 int32_t *__restrict__ pcell, unsigned int *__restrict__ count) {
  const int i = begin + blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= end) return;
  const bool fly = flying ? (flying[i] == 1) : true;
  int32_t c = -1;
  if (fly) {
    double x, y, z;
    if (origin) {
      x = origin[3 * (size_t)i]; y = origin[3 * (size_t)i + 1]; z = origin[3 * (size_t)i + 2];
    } else {
      const ParticleState s = load_state(state + i);
      x = s.x; y = s.y; z = s.z;
    }
    c = cell_of(g, x, y, z);
    atomicAdd(count + c, 1u);
  }
  pcell[i] = c;
}

// exclusive scan of count[0..n) in three small kernels (n <= 2^24)
__global__ void scan_block_kernel(unsigned int *__restrict__ data, unsigned int *__restrict__ sums, int n) {
  __shared__ unsigned int warp_tot[8];
  const int base = blockIdx.x * kScanBlock + threadIdx.x * 4;
  unsigned int v[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) v[k] = (base + k < n) ? data[base + k] : 0u;
  const unsigned int mine = v[0] + v[1] + v[2] + v[3];
  unsigned int inc = mine;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const unsigned int t = __shfl_up_sync(0xffffffffu, inc, d);
    if (lane >= d) inc += t;
  }
  if (lane == 31) warp_tot[warp] = inc;
  __syncthreads();
  unsigned int off = 0;
  for (int w = 0; w < warp; ++w) off += warp_tot[w];
  unsigned int run = off + inc - mine;  // exclusive prefix of this thread within the block
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    if (base + k < n) data[base + k] = run;
    run += v[k];
  }
  if (threadIdx.x == 255) sums[blockIdx.x] = off + inc;
}

__global__ void scan_sums_kernel(unsigned int *__restrict__ sums, int nb, unsigned int *__restrict__ total) {
  // single block: serial over tiles of 1024 block sums (nb <= 16384)
  __shared__ unsigned int carry;
  __shared__ unsigned int warp_tot[32];
  if (threadIdx.x == 0) carry = 0;
  __syncthreads();
  for (int t0 = 0; t0 < nb; t0 += 1024) {
    const int i = t0 + threadIdx.x;
    const unsigned int v = i < nb ? sums[i] : 0u;
    unsigned int inc = v;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const unsigned int t = __shfl_up_sync(0xffffffffu, inc, d);
      if (lane >= d) inc += t;
    }
    if (lane == 31) warp_tot[warp] = inc;
    __syncthreads();
    unsigned int off = carry;
    for (int w = 0; w < warp; ++w) off += warp_tot[w];
    if (i < nb) sums[i] = off + inc - v;
    __syncthreads();
    if (threadIdx.x == 1023) carry = off + inc;
    __syncthreads();
  }
  if (threadIdx.x == 0) *total = carry;
}

__global__ void scan_add_kernel(unsigned int *__restrict__ data, const unsigned int *__restrict__ sums, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) data[i] += sums[i / kScanBlock];
}

// pass 2: scatter particle ids into their cell's slot range (cursor = scanned histogram)
__global__ void bin_scatter_kernel(const int32_t *__restrict__ pcell, int32_t begin, int32_t end,
                                   unsigned int *__restrict__ cursor, int32_t *__restrict__ order) {
  const int i = begin + blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= end) return;
  const int32_t c = pcell[i];
  if (c >= 0) order[atomicAdd(cursor + c, 1u)] = i;
}

// pass 2, packed flavour: the particle's inputs and parent element go to its slot as one 64-byte row
__global__ void bin_pack_kernel(const int32_t *__restrict__ pcell, int32_t begin, int32_t end,
                                unsigned int *__restrict__ cursor, const double *__restrict__ origin,
                                const double *__restrict__ dest, const double *__restrict__ weights,
                                const ParticleState *__restrict__ state, PackedRow *__restrict__ rows) {
  const int i = begin + blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= end) return;
  const int32_t c = pcell[i];
  if (c < 0) return;
  const ParticleState s = load_state(state + i);
  const double ox = origin ? origin[3 * (size_t)i] : s.x, oy = origin ? origin[3 * (size_t)i + 1] : s.y,
               oz = origin ? origin[3 * (size_t)i + 2] : s.z;
  const double dx = dest[3 * (size_t)i], dy = dest[3 * (size_t)i + 1], dz = dest[3 * (size_t)i + 2];
  const double w = weights[i];
  const bool moved = ox != s.x || oy != s.y || oz != s.z;  // same test as begin_particle()
  const unsigned long long tail = (unsigned long long)(uint32_t)i |
                                  ((unsigned long long)(((uint32_t)s.elem & kIdMask) | (moved ? 0x80000000u : 0u)) << 32);
  PackedRow *row = rows + atomicAdd(cursor + c, 1u);
  asm volatile("st.global.L1::no_allocate.v4.b64 [%0], {%1,%2,%3,%4};" ::"l"(row),
               "l"(__double_as_longlong(ox)), "l"(__double_as_longlong(oy)), "l"(__double_as_longlong(oz)),
               "l"(__double_as_longlong(dx))
               : "memory");
  asm volatile("st.global.L1::no_allocate.v4.b64 [%0], {%1,%2,%3,%4};" ::"l"(reinterpret_cast<char *>(row) + 32),
               "l"(__double_as_longlong(dy)), "l"(__double_as_longlong(dz)), "l"(__double_as_longlong(w)), "l"(tail)
               : "memory");
}

}  // namespace

cudaError_t launch_bin_pack_particles(const SeedGrid &g, const double *origin, const double *dest,
                                      const double *weights, const int8_t *flying, const ParticleState *state,
                                      int32_t begin, int32_t end, int32_t *pcell, unsigned int *count,
                                      unsigned int *sums, PackedRow *rows, unsigned int *work_count,
                                      cudaStream_t stream) {
  const int32_t ncell = g.nx * g.ny * g.nz;
  const int n = end - begin;
  if (n <= 0) return cudaMemsetAsync(work_count, 0, sizeof(unsigned int), stream);
  cudaError_t e = cudaMemsetAsync(count, 0, size_t(ncell) * sizeof(unsigned int), stream);
  if (e != cudaSuccess) return e;
  bin_count_kernel<<<(n + 255) / 256, 256, 0, stream>>>(g, origin, state, flying, begin, end, pcell, count);
  const int nb = (ncell + kScanBlock - 1) / kScanBlock;
  scan_block_kernel<<<nb, 256, 0, stream>>>(count, sums, ncell);
  scan_sums_kernel<<<1, 1024, 0, stream>>>(sums, nb, work_count);
  scan_add_kernel<<<(ncell + 255) / 256, 256, 0, stream>>>(count, sums, ncell);
  bin_pack_kernel<<<(n + 255) / 256, 256, 0, stream>>>(pcell, begin, end, count, origin, dest, weights, state, rows);
  return cudaGetLastError();
}

// count: [ncell] scratch (zeroed here), sums: [ceil(ncell/1024)] scratch, order: [end-begin]
// compact output, work_count: device scalar receiving the number of flying particles.
cudaError_t launch_bin_particles(const SeedGrid &g, const double *origin, const ParticleState *state,
                                 const int8_t *flying, int32_t begin, int32_t end, int32_t *pcell, unsigned int *count,
                                 unsigned int *sums, int32_t *order, unsigned int *work_count,
                                 cudaStream_t stream) {
  const int32_t ncell = g.nx * g.ny * g.nz;
  const int n = end - begin;
  if (n <= 0) return cudaMemsetAsync(work_count, 0, sizeof(unsigned int), stream);
  cudaError_t e = cudaMemsetAsync(count, 0, size_t(ncell) * sizeof(unsigned int), stream);
  if (e != cudaSuccess) return e;
  bin_count_kernel<<<(n + 255) / 256, 256, 0, stream>>>(g, origin, state, flying, begin, end, pcell, count);
  const int nb = (ncell + kScanBlock - 1) / kScanBlock;
  scan_block_kernel<<<nb, 256, 0, stream>>>(count, sums, ncell);
  scan_sums_kernel<<<1, 1024, 0, stream>>>(sums, nb, work_count);
  scan_add_kernel<<<(ncell + 255) / 256, 256, 0, stream>>>(count, sums, ncell);
  bin_scatter_kernel<<<(n + 255) / 256, 256, 0, stream>>>(pcell, begin, end, count, order);
  return cudaGetLastError();
}

}  // namespace ptb
