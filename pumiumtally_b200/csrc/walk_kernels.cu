// sm_100a kernels of the track-length tally engine: the kernels the engine chooses between.
//
// One fused kernel per particle range does what the reference spreads over
// K1..K12 of SURVEY.md section 2b: the "set dest" kernels
// (PumiTallyImpl.cpp:88-109, 127-142, 186-192), both SearchAndRebuild loops
// (PumiTallyImpl.cpp:433-459 -> external tracer) and the per-iteration functor
// (PumiTallyImpl.cpp:297-316).  Each particle is walked to completion in
// registers; the only global traffic per crossing is three 32-byte sectors of
// one tet record and one fp64 reduction into flux[elem].
//
// Product variants (WalkVariant in walk_kernels.hpp): 0 thread per particle (first correct path,
// kept as the in-library cross-check), 8 persistent streaming kernel (default, mesh <~ 2x L2),
// 16 persistent kernel on spatially binned particles (default, mesh >> L2), 24 persistent kernel
// on packed sorted rows (picked by the auto-tuner for collimated long tracks).  Every other
// variant number is a measured alternative that lives in experiments/walk_experiments.cu and is
// only linked into libpumitally_exp.so (build flag PTB_EXPERIMENTS).
#include "walk_kernels.hpp"

#include "walk_persist.cuh"

namespace ptb {
namespace {

// ---------------------------------------------------------------- variant 0
// Thread per particle; the 128-byte record arrives as four 256-bit loads
// (LDG.E.ENL2.256), one per face.

__global__ void __launch_bounds__(256) walk_ldg_kernel(const WalkParams P) {
  const int i = P.begin + blockIdx.x * blockDim.x + threadIdx.x;
  Counters c;
  Ray r;
  r.stage = kStageDone;
  if (i < P.end) begin_particle(P, i, r, c, true);
  while (r.stage != kStageDone) {
    const double *rec = P.tets[r.e].d;
    double raw[16];
#pragma unroll
    for (int f = 0; f < 4; ++f)
      load_face_256(rec + 4 * f, raw[4 * f], raw[4 * f + 1], raw[4 * f + 2], raw[4 * f + 3]);
    ExitScan sc;
    scan_record(raw, r.e, r.ox, r.oy, r.oz, r.ux, r.uy, r.uz, sc);
    advance(P, i, r, exit_parameter(sc), sc.nbr, sc.back, c, true);
  }
  flush_counters(P, c);
}

// ------------------------------------------------------------ small kernels

// K14-K16 of SURVEY.md 2b (PumiTallyImpl.cpp:492-528): every particle starts
// at the centroid of element 0.
__global__ void init_particles_kernel(ParticleState *state, int32_t n, double cx, double cy, double cz,
                                      int32_t elem) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) store_state(state + i, cx, cy, cz, elem);
}

// Seed grid construction: the seed points are written as "particles to
// localise", walked with the ordinary kernel, and a cell keeps the tet only if
// its seed point was reached (i.e. lies inside the mesh).
__global__ void seed_points_kernel(SeedGrid g, double *xyz, int32_t ncell) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < ncell) {
    const int cx = i % g.nx, cy = (i / g.nx) % g.ny, cz = i / (g.nx * g.ny);
    double x, y, z;
    seed_point(g, cx, cy, cz, x, y, z);
    xyz[3 * (size_t)i] = x; xyz[3 * (size_t)i + 1] = y; xyz[3 * (size_t)i + 2] = z;
  }
}

__global__ void seed_finalize_kernel(const double *xyz, const ParticleState *state, int32_t *cell_tet,
                                     int32_t ncell) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < ncell) {
    const ParticleState s = load_state(state + i);
    const bool reached = s.x == xyz[3 * (size_t)i] && s.y == xyz[3 * (size_t)i + 1] && s.z == xyz[3 * (size_t)i + 2];
    cell_tet[i] = reached ? s.elem : -1;
  }
}

// Delta upload of the host-pointer path: the origin array on the device starts as the previous
// move's destinations; only the particles whose caller-side origin differs are patched.
__global__ void patch_origins_kernel(double *origin, const PatchEntry *list, int32_t count) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= count) return;
  double x, y, z, w;
  load_face_256(reinterpret_cast<const double *>(list + i), x, y, z, w);
  const int32_t idx = (int32_t)((unsigned long long)__double_as_longlong(w) & 0xffffffffull);
  origin[3 * (size_t)idx] = x;
  origin[3 * (size_t)idx + 1] = y;
  origin[3 * (size_t)idx + 2] = z;
}

// Particle slots [begin, end) <- (xyz, element in the caller's numbering): for callers that manage
// particle placement themselves (the spatially partitioned multi-GPU driver hands particles from one
// picpart to the next).  elem_map: caller's element id -> internal id.
__global__ void set_state_kernel(ParticleState *state, const double *xyz, const int32_t *elem, const int32_t *elem_map,
                                 int32_t begin, int32_t end) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  const int i = begin + k;
  if (i >= end) return;
  store_state(state + i, xyz[3 * (size_t)k], xyz[3 * (size_t)k + 1], xyz[3 * (size_t)k + 2], elem_map[elem[k]]);
}

// (xyz, element in the caller's numbering) <- particle slots [begin, end).  elem_map: internal id -> caller's.
__global__ void get_state_kernel(const ParticleState *state, double *xyz, int32_t *elem, const int32_t *elem_map,
                                 int32_t begin, int32_t end) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  const int i = begin + k;
  if (i >= end) return;
  const ParticleState s = load_state(state + i);
  xyz[3 * (size_t)k] = s.x;
  xyz[3 * (size_t)k + 1] = s.y;
  xyz[3 * (size_t)k + 2] = s.z;
  elem[k] = elem_map[s.elem];
}

// out[caller's element id] = flux[internal id]
__global__ void flux_to_caller_order_kernel(const double *flux, const int32_t *orig_of_internal, double *out, int64_t n) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e < n) out[orig_of_internal[e]] = flux[e];
}

// K13 (PumiTallyImpl.cpp:393-405) with volumes precomputed at mesh build.
__global__ void normalize_kernel(const double *flux, const double *volume, double *out, int64_t n, double per_source) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e < n) out[e] = flux[e] / volume[e] / per_source;  // per_source == 1: bit-identical to flux / volume
}

// Score filter (engine.cu, launch_range): the flying flags of the particles whose score bin is `bin`
// (bin == nbins: of those whose bin is outside [0, nbins) -- they fly, unscored)
__global__ void bin_mask_kernel(const int8_t *flying, const int32_t *bins, int32_t bin, int32_t nbins, int8_t *mask,
                                int32_t begin, int32_t end) {
  const int i = begin + (int)(blockIdx.x * blockDim.x + threadIdx.x);
  if (i >= end) return;
  const int32_t b = bins[i];
  const bool mine = (b >= 0 && b < nbins) ? b == bin : bin == nbins;
  mask[i] = (mine && (!flying || flying[i] == 1)) ? 1 : 0;
}

// Total weight of the particles that fly in this range (the reference's total_initial_weight,
// PumiTallyImpl.h:170-171: declared "needed for normalization", never filled in).
__global__ void sum_flying_weights_kernel(const int8_t *flying, const double *weights, int32_t begin, int32_t end,
                                          double *total) {
  double s = 0.0;
  for (int i = begin + blockIdx.x * blockDim.x + threadIdx.x; i < end; i += gridDim.x * blockDim.x)
    if ((!flying || flying[i] == 1) && all_finite(weights[i], 0.0, 0.0)) s += weights[i];
  for (int d = 16; d > 0; d >>= 1) s += __shfl_down_sync(0xffffffffu, s, d);
  if ((threadIdx.x & 31) == 0 && s != 0.0) atomicAdd(total, s);
}

}  // namespace

#ifdef PTB_EXPERIMENTS
cudaError_t launch_walk_experiment(const WalkParams &p, int variant, int block, cudaStream_t stream);
#endif

cudaError_t launch_walk(const WalkParams &p, int variant, int block, cudaStream_t stream) {
  const long long n = (long long)p.end - p.begin;
  if (n <= 0) return cudaSuccess;
  if (block != 64 && block != 128 && block != 256) block = 128;
  switch (variant) {
    case kVariantLdg: {
      const unsigned grid = (unsigned)((n + block - 1) / block);
      walk_ldg_kernel<<<grid, block, 0, stream>>>(p);
      return cudaGetLastError();
    }
    case kVariantPersistRefill8:
      return launch_persist<128, kFetchPolicy, 7, 8>(p, n, stream);
    case kVariantPersistGatherL1:
      return launch_persist<128, kFetchPolicyL1, 6, 8, true, 40>(p, n, stream);
    case kVariantPacked:
      if (!p.rows) return cudaErrorInvalidValue;
      return launch_persist<128, kFetchPolicy, 7, 8, 2>(p, n, stream);
    default:
#ifdef PTB_EXPERIMENTS
      return launch_walk_experiment(p, variant, block, stream);
#else
      return cudaErrorInvalidValue;
#endif
  }
}

bool walk_variant_available(int variant) {
  switch (variant) {
    case kVariantLdg: case kVariantPersistRefill8: case kVariantPersistGatherL1: case kVariantPacked:
      return true;
    default:
#ifdef PTB_EXPERIMENTS
      return variant >= 0 && variant < kNumVariants;
#else
      return false;
#endif
  }
}

cudaError_t launch_init_particles(ParticleState *state, int32_t n, double cx, double cy, double cz,
                                  int32_t elem, cudaStream_t stream) {
  if (n <= 0) return cudaSuccess;
  init_particles_kernel<<<(n + 255) / 256, 256, 0, stream>>>(state, n, cx, cy, cz, elem);
  return cudaGetLastError();
}

cudaError_t launch_seed_points(const SeedGrid &g, double *xyz, cudaStream_t stream) {
  const int32_t ncell = g.nx * g.ny * g.nz;
  seed_points_kernel<<<(ncell + 255) / 256, 256, 0, stream>>>(g, xyz, ncell);
  return cudaGetLastError();
}

cudaError_t launch_seed_finalize(const double *xyz, const ParticleState *state, int32_t *cell_tet,
                                 int32_t ncell, cudaStream_t stream) {
  seed_finalize_kernel<<<(ncell + 255) / 256, 256, 0, stream>>>(xyz, state, cell_tet, ncell);
  return cudaGetLastError();
}

cudaError_t launch_patch_origins(double *origin, const PatchEntry *list, int32_t count, cudaStream_t stream) {
  if (count <= 0) return cudaSuccess;
  patch_origins_kernel<<<(count + 255) / 256, 256, 0, stream>>>(origin, list, count);
  return cudaGetLastError();
}

cudaError_t launch_set_state(ParticleState *state, const double *xyz, const int32_t *elem, const int32_t *elem_map,
                             int32_t begin, int32_t end, cudaStream_t stream) {
  if (end <= begin) return cudaSuccess;
  set_state_kernel<<<(end - begin + 255) / 256, 256, 0, stream>>>(state, xyz, elem, elem_map, begin, end);
  return cudaGetLastError();
}

cudaError_t launch_get_state(const ParticleState *state, double *xyz, int32_t *elem, const int32_t *elem_map,
                             int32_t begin, int32_t end, cudaStream_t stream) {
  if (end <= begin) return cudaSuccess;
  get_state_kernel<<<(end - begin + 255) / 256, 256, 0, stream>>>(state, xyz, elem, elem_map, begin, end);
  return cudaGetLastError();
}

cudaError_t launch_flux_to_caller_order(const double *flux, const int32_t *orig_of_internal, double *out, int64_t n,
                                        cudaStream_t stream) {
  if (n <= 0) return cudaSuccess;
  flux_to_caller_order_kernel<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(flux, orig_of_internal, out, n);
  return cudaGetLastError();
}

cudaError_t launch_normalize(const double *flux, const double *volume, double *out, int64_t n,
                             double per_source, cudaStream_t stream) {
  if (n <= 0) return cudaSuccess;
  normalize_kernel<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(flux, volume, out, n, per_source);
  return cudaGetLastError();
}

cudaError_t launch_bin_mask(const int8_t *flying, const int32_t *bins, int32_t bin, int32_t nbins, int8_t *mask,
                            int32_t begin, int32_t end, cudaStream_t stream) {
  if (end <= begin) return cudaSuccess;
  bin_mask_kernel<<<(end - begin + 255) / 256, 256, 0, stream>>>(flying, bins, bin, nbins, mask, begin, end);
  return cudaGetLastError();
}

cudaError_t launch_sum_flying_weights(const int8_t *flying, const double *weights, int32_t begin, int32_t end,
                                      double *total, cudaStream_t stream) {
  if (end <= begin) return cudaSuccess;
  const int n = end - begin;
  sum_flying_weights_kernel<<<std::min((n + 255) / 256, 1184), 256, 0, stream>>>(flying, weights, begin, end, total);
  return cudaGetLastError();
}

}  // namespace ptb