// Additive calls for code that uses pumitally::PumiTally (the reference class, whose header ships
// unchanged because it is the ABI) and wants what the reference left as TODOs: tally reset between
// batches and per-source-particle normalisation (reference: PumiTally.h:93 "Normalized by element
// volumes and total number of particles" vs PumiTallyImpl.cpp:402 which divides by volume only;
// total_initial_weight, PumiTallyImpl.h:170-171, declared and never used).
//
// engine_of() hands out the C-ABI handle behind a PumiTally object; everything in pumitally_c.h can
// be used on it (pumitally_reset_tally, pumitally_set_source_normalization, pumitally_get_flux,
// pumitally_comm_init / pumitally_allreduce_tally for several GPUs, ...).
#ifndef PUMITALLY_PUMITALLYEXTRAS_H
#define PUMITALLY_PUMITALLYEXTRAS_H

#include "pumitally/PumiTally.h"
#include "pumitally_c.h"

namespace pumitally {

// nullptr if `tally` is not a live PumiTally object
pumitally_engine *engine_of(const PumiTally &tally);

// Start over: zero the flux, the statistics, the batch statistics and the initial-track weight.
inline int ResetTally(const PumiTally &tally) { return pumitally_reset_tally(engine_of(tally)); }

// mode 0 volume only (reference behaviour), 1 / num_particles, 2 / value, 3 / total weight of the
// batch's first tracks (see pumitally_set_source_normalization).
inline int SetSourceNormalization(const PumiTally &tally, int mode, double value = 1.0) {
  return pumitally_set_source_normalization(engine_of(tally), mode, value);
}

// Score filter: `nbins` flux arrays; MoveToNextLocationBinned scores particle i into array bins[i]
// (see pumitally_set_score_bins in pumitally_c.h).
inline int SetScoreBins(const PumiTally &tally, int32_t nbins) { return pumitally_set_score_bins(engine_of(tally), nbins); }
inline int MoveToNextLocationBinned(const PumiTally &tally, double *particle_origin, double *particle_destinations,
                                    int8_t *flying, double *weights, const int32_t *bins, int32_t size) {
  return pumitally_move_to_next_location_binned(engine_of(tally), particle_origin, particle_destinations, flying,
                                                weights, bins, size);
}

// Batch statistics (see pumitally_end_batch in pumitally_c.h): close the batch, read mean and standard
// deviation of the mean per element (n = num_elements or nbins * num_elements), query the relative-error
// trigger.  Collective on several GPUs.
inline int EndBatch(const PumiTally &tally) { return pumitally_end_batch(engine_of(tally)); }
inline int GetTallyStatistics(const PumiTally &tally, double *mean, double *std_dev, int64_t n) {
  return pumitally_get_tally_statistics(engine_of(tally), mean, std_dev, n);
}
inline int MaxRelativeError(const PumiTally &tally, double threshold, double *max_rel, int64_t *index,
                            int64_t *count_above) {
  return pumitally_get_max_relative_error(engine_of(tally), threshold, max_rel, index, count_above);
}

}  // namespace pumitally

#endif  // PUMITALLY_PUMITALLYEXTRAS_H
