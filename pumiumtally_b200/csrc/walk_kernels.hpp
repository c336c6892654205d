// Launch interface of the sm_100a walk/tally kernels (walk_kernels.cu).
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#include "tet_mesh.hpp"
#include "walk_core.cuh"

namespace ptb {

// Values are stable (profiles/ refer to them); the gaps are experiments that were measured,
// lost and removed (9/10 other refill thresholds, 11/12/14 cooperative transposed fetch, 18).
// libpumitally.so contains the four kernels the engine chooses between -- 0, 8, 16, 24; the other
// numbers are measured alternatives compiled only into libpumitally_exp.so
// (experiments/walk_experiments.cu, build flag PTB_EXPERIMENTS).
enum WalkVariant : int {
  kVariantLdg = 0,    // thread per particle, 4 x 256-bit loads of the tet record (first correct path)
  kVariantBulk = 1,   // thread per particle, record staged in smem by cp.async.bulk + mbarrier
  kVariantQuad = 2,   // 4 lanes per particle (lane per face), coalesced 32 B loads
  kVariantPersist = 3,               // persistent warps, TMA-staged particle chunks, per-lane refill
  kVariantPersistPolicy = 4,         // 3 + L2 evict_last on tets / evict_first on the particle stream
  kVariantPersistPolicy128 = 5,      // 4 + L2::128B prefetch size on tet loads
  kVariantPersistBulk = 6,           // 4 with tet records fetched by cp.async.bulk into smem rows
  kVariantPersistPolicy128Occ8 = 7,  // 5 compiled for 8 resident blocks (64 registers)
  kVariantPersistRefill8 = 8,        // 4, refilling only when >= 8 lanes are idle (default, mesh <~ 2x L2)
  kVariantPersistRefill8Occ8 = 9,    // 8 compiled for 8 resident blocks (64 registers) -- re-test after entry-face elision
  kVariantPersistBulkOcc7 = 13,      // 6 compiled for 7 resident blocks
  kVariantPersistGather = 15,        // 8 on spatially binned particles (order[] from launch_bin_particles)
  kVariantPersistGatherL1 = 16,      // 15 with L1-allocating tet loads (default, mesh >> L2)
  kVariantPersistGatherPlain = 17,   // 15 with plain tet loads (no L2 policy)
  kVariantEdge = 20,        // compact layout + edge-function exit test (walk_compact.cuh), streaming order
  kVariantEdgeGather = 21,  // 20 on spatially binned particles
  kVariantEdgeOcc5 = 22,    // 20 compiled for 5 resident blocks (96 registers, a few spills)
  kVariantEdgeOcc6 = 23,    // 20 compiled for 6 resident blocks (80 registers, more spills)
  kVariantPacked = 24,      // 8 on a packed, spatially sorted copy of the flying particles' inputs (bin + pack pass)
  kVariantPackedL1 = 25,    // 24 with L1-allocating tet loads (neighbouring lanes share records once particles are sorted)
  kVariantPackedL1Occ6 = 26,
  kVariantTwoRays = 27,        // 8 with two rays per lane in flight (software-pipelined walk)
  kVariantPersistAggTally = 28,  // 8 with the warp-aggregated tally (match.any + shuffles)
  kVariantGatherAggTally = 29,   // 16 with the warp-aggregated tally
  kVariantLean = 30,        // 8 with the lean crossing step (three loads as one block, payload decoded once, target re-read)
  kVariantLeanGather = 31,  // 16 with the lean crossing step
  kVariantLeanPacked = 32,  // 24 with the lean crossing step
  kNumVariants = 33
};

// how a variant gets its particles: through order[] from the binning pass / through packed rows
inline bool variant_is_gather(int v) {
  return v == kVariantPersistGather || v == kVariantPersistGatherL1 || v == kVariantPersistGatherPlain ||
         v == kVariantEdgeGather || v == kVariantGatherAggTally || v == kVariantLeanGather;
}
inline bool variant_is_packed(int v) {
  return v == kVariantPacked || v == kVariantPackedL1 || v == kVariantPackedL1Occ6 || v == kVariantLeanPacked;
}


cudaError_t launch_walk(const WalkParams &p, int variant, int block, cudaStream_t stream);
bool walk_variant_available(int variant);  // compiled into this library?
// origin == nullptr: the binning key is the stored position (state)
cudaError_t launch_bin_particles(const SeedGrid &g, const double *origin, const ParticleState *state,
                                 const int8_t *flying, int32_t begin, int32_t end, int32_t *pcell, unsigned int *count,
                                 unsigned int *sums, int32_t *order, unsigned int *work_count,
                                 cudaStream_t stream);
// Like launch_bin_particles, but instead of the id list the scatter pass writes one PackedRow per
// flying particle (origin, dest, weight, id, parent element + relocate flag) in cell order.
cudaError_t launch_bin_pack_particles(const SeedGrid &g, const double *origin, const double *dest,
                                      const double *weights, const int8_t *flying, const ParticleState *state,
                                      int32_t begin, int32_t end, int32_t *pcell, unsigned int *count,
                                      unsigned int *sums, PackedRow *rows, unsigned int *work_count,
                                      cudaStream_t stream);
cudaError_t launch_seed_points(const SeedGrid &g, double *xyz, cudaStream_t stream);
cudaError_t launch_seed_finalize(const double *xyz, const ParticleState *state, int32_t *cell_tet,
                                 int32_t ncell, cudaStream_t stream);
cudaError_t launch_init_particles(ParticleState *state, int32_t n, double cx, double cy, double cz,
                                  int32_t elem, cudaStream_t stream);
// origin[3*idx..] = (x,y,z) for every entry of the patch list
cudaError_t launch_patch_origins(double *origin, const PatchEntry *list, int32_t count, cudaStream_t stream);
// particle slots [begin, end) <-> (xyz[3k..], elem[k]) with k = slot - begin; elem in the caller's numbering
cudaError_t launch_set_state(ParticleState *state, const double *xyz, const int32_t *elem, const int32_t *elem_map,
                             int32_t begin, int32_t end, cudaStream_t stream);
cudaError_t launch_get_state(const ParticleState *state, double *xyz, int32_t *elem, const int32_t *elem_map,
                             int32_t begin, int32_t end, cudaStream_t stream);
cudaError_t launch_flux_to_caller_order(const double *flux, const int32_t *orig_of_internal, double *out, int64_t n,
                                        cudaStream_t stream);
// out = flux / volume / per_source (NormalizeFlux, PumiTallyImpl.cpp:393-405; per_source = 1 is the reference)
cudaError_t launch_normalize(const double *flux, const double *volume, double *out, int64_t n,
                             double per_source, cudaStream_t stream);

// mask[i] = flying[i] && bins[i] == bin  (bin == nbins selects the particles outside [0, nbins))
cudaError_t launch_bin_mask(const int8_t *flying, const int32_t *bins, int32_t bin, int32_t nbins, int8_t *mask,
                            int32_t begin, int32_t end, cudaStream_t stream);
// *total += sum of weights[i] over flying particles of [begin, end)
cudaError_t launch_sum_flying_weights(const int8_t *flying, const double *weights, int32_t begin, int32_t end,
                                      double *total, cudaStream_t stream);

}  // namespace ptb
