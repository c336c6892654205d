/*
 * pumitally_c.h -- C ABI of libpumitally.so (B200 track-length tally engine).
 *
 * Plain pointers and sizes only.  The first five entry points are one-to-one
 * with the reference's public interface, which is what any FFI for this path
 * binds (reference: src/pumitally/PumiTally.h, class pumitally::PumiTally);
 * the C++ facade in include/pumitally/PumiTally.h is a thin wrapper over them.
 * The rest are additive: accessors the reference's tests obtain by reaching
 * into PumiTallyImpl members, device-pointer entry points for callers whose
 * particle data already lives in HBM, and the multi-GPU exchange step.
 *
 * Error convention follows the reference (PumiTallyImpl.cpp:444-458, 558-565):
 * problems are printed to stderr and the call returns; functions that return
 * int give 0 on success and non-zero on failure so FFI callers can also check.
 * There is no CPU fallback: without a CUDA device pumitally_create* fails.
 */
#ifndef PUMITALLY_C_H
#define PUMITALLY_C_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct pumitally_engine pumitally_engine;

/* ---- reference interface ------------------------------------------------ */

/* PumiTally::PumiTally(mesh_filename, num_particles, argc, argv)
 * (reference: PumiTally.h:50-51, PumiTallyImpl.cpp:31-52).  mesh_filename: an
 * Omega_h "<name>.osh" directory, a raw mesh file, or "box:nx,ny,nz[,lx,ly,lz]".
 * argc/argv may be NULL.  Returns NULL on failure. */
pumitally_engine *pumitally_create(const char *mesh_filename, int32_t num_particles,
                                   int *argc, char ***argv);

/* PumiTally::CopyInitialPosition(init_particle_positions, size)
 * (reference: PumiTally.h:66-67, PumiTallyImpl.cpp:54-64).  Host pointer,
 * x0,y0,z0,x1,...; size = 3 * num_particles.  Once per engine. */
int pumitally_copy_initial_position(pumitally_engine *e, const double *init_particle_positions,
                                    int32_t size);

/* PumiTally::MoveToNextLocation(origin, destinations, flying, weights, size)
 * (reference: PumiTally.h:87-89, PumiTallyImpl.cpp:66-149).  Host pointers;
 * size = 3 * num_particles; flying[] is overwritten with zeros
 * (PumiTallyImpl.cpp:169-172).  Inputs are fully consumed before return. */
int pumitally_move_to_next_location(pumitally_engine *e, const double *particle_origin,
                                    const double *particle_destinations, int8_t *flying,
                                    const double *weights, int32_t size);

/* PumiTally::WriteTallyResults() (reference: PumiTally.h:95,
 * PumiTallyImpl.cpp:151-157, 382-416): flux/volume -> "fluxresult.vtk". */
int pumitally_write_tally_results(pumitally_engine *e);

/* PumiTally::~PumiTally() (reference: PumiTally.h:103, PumiTally.cpp:16-19). */
void pumitally_destroy(pumitally_engine *e);

/* ---- additive: construction from arrays ---------------------------------- */

/* Same engine, mesh given in memory: coords double[3*nverts], tet2vert
 * int32[4*ntets] (what the reference gets from Omega_h::binary::read,
 * PumiTallyImpl.cpp:562).  device < 0 selects the current CUDA device. */
pumitally_engine *pumitally_create_from_arrays(const double *coords, int64_t nverts,
                                               const int32_t *tet2vert, int64_t ntets,
                                               int32_t num_particles, int32_t device);

/* ---- additive: accessors (reference tests read Impl members instead:
 * test_pumi_tally_impl_methods.cpp:153, 163, 232) ------------------------- */

int64_t pumitally_num_elements(const pumitally_engine *e);
int32_t pumitally_num_particles(const pumitally_engine *e);
/* raw (un-normalised) flux, double[num_elements] (handler->flux); with score bins also
 * n = nbins * num_elements, see pumitally_set_score_bins */
int pumitally_get_flux(pumitally_engine *e, double *out, int64_t n);
/* flux / volume and volume (NormalizeFlux, PumiTallyImpl.cpp:382-409); either may be NULL */
int pumitally_get_normalized_flux(pumitally_engine *e, double *out_flux, double *out_volume,
                                  int64_t n);
/* parent element of every particle, int32[num_particles] (tracer->getElementIds()) */
int pumitally_get_element_ids(pumitally_engine *e, int32_t *out, int64_t n);
/* current particle positions, double[3*num_particles] AoS (ptcls->get<0>()) */
int pumitally_get_positions(pumitally_engine *e, double *out, int64_t n3);
/* face adjacency derived by the engine, int32[4*num_elements], -1 = hull */
int pumitally_get_adjacency(const pumitally_engine *e, int32_t *out, int64_t n4);
/* zero the flux and the statistics (new batch) */
int pumitally_reset_tally(pumitally_engine *e);
/* Per-source-particle normalisation of the NORMALISED flux (pumitally_get_normalized_flux and
 * WriteTallyResults; the raw flux is unaffected).  The reference divides by tet volume only
 * (PumiTallyImpl.cpp:402) although PumiTally.h:93 promises "and total number of particles", and
 * carries an unused total_initial_weight "needed for normalization" (PumiTallyImpl.h:170-171).
 * mode 0: volume only (default = the reference's behaviour); 1: also by num_particles;
 * 2: also by `value` (> 0, e.g. the total source weight of the batch); 3: also by the total weight
 * of the first tracks after CopyInitialPosition / pumitally_reset_tally, summed by the engine. */
int pumitally_set_source_normalization(pumitally_engine *e, int32_t mode, double value);
/* the divisor currently in effect (1.0 for mode 0) */
double pumitally_get_source_normalization(pumitally_engine *e);

typedef struct pumitally_stats {
  uint64_t segments;      /* tally contributions issued in weighted phases (the metric's unit) */
  uint64_t tracks;        /* flying particles in weighted phases */
  uint64_t relocations;   /* tet crossings walked with tallying off (phase 1 + localisation) */
  uint64_t lost;          /* walks stopped by the iteration limit */
  uint64_t moves;         /* MoveToNextLocation calls */
  double kernel_ms;       /* device time of the walk kernels (CUDA events), cumulative */
  double h2d_bytes;       /* bytes uploaded by the host-pointer entry points, cumulative */
  uint64_t plane_fallbacks; /* compact-layout walk: rays coplanar with a mesh edge, finished on the plane records */
} pumitally_stats;
int pumitally_get_stats(pumitally_engine *e, pumitally_stats *out);

/* Per-call output file name for WriteTallyResults (default "fluxresult.vtk"). */
int pumitally_set_output_name(pumitally_engine *e, const char *filename);
/* Options: "variant" (-1 = the engine picks the walk kernel from the mesh size, the default; 0, 8,
 * 16, 24 = the kernels of this library), "block", "chunk" (particles per upload/compute pipeline
 * stage), "seed_grid", "morton", "claim_run", "host_path" (1 = host-pointer moves are staged
 * through pinned per-particle slots by a small worker pool and only the origins that differ from
 * the previous call's destinations travel; 0 = direct copies of all four arrays from the caller's
 * memory; 2 = default: staged, except that for page-locked caller arrays the engine times both and
 * keeps the faster), "host_threads" (workers of that pool, before the first host-pointer call;
 * default: CPU quota / ranks per node - 1; environment: PUMITALLY_HOST_THREADS,
 * PUMITALLY_HOST_PIN=0 keeps them off the GPU's NUMA node), "register_host" (direct path only:
 * 1 = page-lock the caller's pageable buffers with cudaHostRegister the first time they are
 * seen; the caller must then keep them alive; also PUMITALLY_REGISTER_HOST=1), "max_iters"
 * (crossing limit per walk; 0 = number of elements + 16, the default), "l2_fetch", "autotune"
 * (1 = default: while "variant" is automatic the engine times the streaming and the sorted/packed
 * kernel on moves 1-4 of every 64 and keeps the faster one).  Read-only: "launches", "staged",
 * "stage_host_us", "stage_sent_bytes", "batches" (see pumitally_end_batch). */
int pumitally_set_option(pumitally_engine *e, const char *name, int64_t value);
int64_t pumitally_get_option(const pumitally_engine *e, const char *name);

/* ---- additive: device-pointer entry points -------------------------------
 * Same semantics as the host versions, but the arrays already live in device
 * memory (AoS positions, int8 flying, double weights).  Work is enqueued on
 * `stream` (a cudaStream_t passed as void*; NULL = the CUDA default stream,
 * which is also what PyTorch's default stream is) and the call returns
 * without synchronising.  d_flying is NOT zeroed. */
int pumitally_copy_initial_position_device(pumitally_engine *e, const double *d_xyz, int32_t size,
                                           void *stream);
int pumitally_move_to_next_location_device(pumitally_engine *e, const double *d_origin,
                                           const double *d_destinations, const int8_t *d_flying,
                                           const double *d_weights, int32_t size, void *stream);
/* Particle slots [first, first+count) <- positions d_xyz[3*count] in elements d_elem[count] (the
 * caller's element numbering), without walking there; and the reverse.  For drivers that place
 * particles themselves, e.g. the spatially partitioned multi-GPU driver
 * (pumiumtally_b200/partition.py), which hands particles from one picpart's engine to the next.
 * The elements are trusted to contain the positions.  Enqueued on `stream`, no synchronisation. */
int pumitally_set_state_device(pumitally_engine *e, const double *d_xyz, const int32_t *d_elem,
                               int32_t first, int32_t count, void *stream);
int pumitally_get_state_device(pumitally_engine *e, double *d_xyz, int32_t *d_elem, int32_t first,
                               int32_t count, void *stream);
/* raw flux in the caller's element numbering into device memory d_out[num_elements] */
int pumitally_get_flux_device(pumitally_engine *e, double *d_out, void *stream);
/* device address of the raw flux array (double[num_elements]); NOTE: in the engine's internal
 * (spatially sorted) element order -- use pumitally_get_flux for the caller's numbering */
double *pumitally_flux_device_ptr(pumitally_engine *e);
int pumitally_synchronize(pumitally_engine *e);

/* ---- additive: multi-GPU exchange step -----------------------------------
 * One engine per GPU/process.  Every rank holds a picpart of the mesh and a
 * slice of the particles; at batch end the per-rank tallies of shared (ghost)
 * elements are summed with ncclAllReduce over NVLink.  The 128-byte unique id
 * is produced on rank 0 and distributed by the caller (MPI_Bcast in OpenMC,
 * torch.distributed in bench.py). */
int pumitally_nccl_unique_id(uint8_t out_id[128]);
int pumitally_comm_init(pumitally_engine *e, int32_t rank, int32_t nranks, const uint8_t id[128]);
int pumitally_allreduce_tally(pumitally_engine *e);
/* The cheaper batch-end exchange (half the NVLink traffic): ncclReduceScatter -- every rank receives
 * the sum over ranks of its own share of the elements only.  The shares are gathered (ncclAllGather,
 * COLLECTIVE: every rank must make the call) the first time pumitally_get_flux,
 * pumitally_get_normalized_flux, pumitally_get_flux_device or pumitally_write_tally_results needs
 * the whole array, i.e. normally once, at the end of the run. */
int pumitally_reduce_tally_to_owners(pumitally_engine *e);
/* Which of the two is quicker depends on the size of the flux array and on the algorithm NCCL picks for
 * it (8 B200s: 8 MB -- all-reduce 0.10 ms, reduce-scatter 4.3 ms; 79 MB -- 0.9 ms and 0.43 ms), so
 * pumitally_comm_init times both on the engine's own mesh, agrees on the result across the ranks, and
 * this call -- the one a driver should make at batch end -- runs the quicker one.  Read the decision
 * with pumitally_get_option("exchange_choice") (0 all-reduce, 1 reduce-scatter) and the two times with
 * "exchange_allreduce_us" / "exchange_reduce_scatter_us". */
int pumitally_exchange_tally(pumitally_engine *e);

/* ---- additive: score filter (SURVEY section 8 f4) ---------------------------
 * The reference tallies one flux array (PumiTallyImpl.h:142, flux[elem] += length * weight,
 * PumiTallyImpl.cpp:376); an OpenMC tally usually carries a filter -- energy group, particle type,
 * material -- that sends a score to one of several bins.  pumitally_set_score_bins(e, nbins)
 * gives the engine nbins flux arrays (and resets the tally; on several GPUs call it before
 * pumitally_comm_init), and the *_binned moves take one more per-particle array: the bin particle i
 * scores into during this move.  A bin outside [0, nbins) means "no bin matches": the particle
 * flies and is clipped like any other, unscored.  bins == NULL or nbins == 1 is the plain move.
 * With nbins > 1, pumitally_get_flux / pumitally_get_normalized_flux accept n = num_elements (bin 0)
 * or n = nbins * num_elements (every bin, bin-major); pumitally_get_flux_device always writes every
 * bin; WriteTallyResults writes "flux" = the sum over the bins plus "flux_bin<k>" per bin; the
 * batch-end exchange moves all bins.  The walk kernels are the unfiltered ones: a binned move walks
 * the particle range once per bin with the flying flags masked to that bin (particles are independent
 * and a particle that does not fly is not touched), so it costs one extra pass over the particle
 * arrays per bin, not per segment. */
int pumitally_set_score_bins(pumitally_engine *e, int32_t nbins);
int32_t pumitally_get_score_bins(const pumitally_engine *e);
int pumitally_move_to_next_location_binned(pumitally_engine *e, const double *particle_origin,
                                           const double *particle_destinations, int8_t *flying,
                                           const double *weights, const int32_t *bins, int32_t size);
int pumitally_move_to_next_location_device_binned(pumitally_engine *e, const double *d_origin,
                                                  const double *d_destinations, const int8_t *d_flying,
                                                  const double *d_weights, const int32_t *d_bins,
                                                  int32_t size, void *stream);

/* ---- additive: batch statistics ------------------------------------------
 * Every Monte Carlo tally result is a mean over batches with the standard deviation of that mean; OpenMC
 * keeps a running sum and sum of squares per bin over the active batches, and its tally triggers stop a
 * run once the relative error falls below a threshold.  pumitally_end_batch closes the current batch:
 * the raw flux since the last end_batch / pumitally_reset_tally / pumitally_set_score_bins /
 * CopyInitialPosition (summed over ranks when a communicator exists, by the exchange pumitally_comm_init
 * chose; an earlier pumitally_exchange_tally result is superseded) is divided by the batch's source
 * divisor -- mode 0: 1; mode 1: the number of particles summed over ranks; mode 2: `value`, the global
 * source weight of one batch; mode 3: the weight of the batch's first tracks summed over ranks -- and the
 * result x is added to S1 and x*x to S2 per (bin, element); then the flux and the first-track weight start
 * over.  A divisor that is not finite and > 0 makes the call fail and change nothing.  pumitally_stats keep
 * counting; pumitally_reset_tally and pumitally_set_score_bins discard S1, S2 and the batch count n
 * (pumitally_get_option "batches").  On several GPUs each rank keeps the sums of its share of the elements
 * (the reduce-scatter layout of pumitally_reduce_tally_to_owners) and all three calls are COLLECTIVE.
 * Moves may be on any stream: end_batch synchronises the device first and returns after its own pass. */
int pumitally_end_batch(pumitally_engine *e);
/* mean = S1 / n / volume and its standard deviation sqrt((S2/n - (S1/n)^2) / (n - 1)) / volume (a negative
 * rounding residue is clamped to 0; NaN with n == 1), caller's element numbering; n as for
 * pumitally_get_flux; either pointer may be NULL.  Fails before the first end_batch.  WriteTallyResults
 * writes the mean as "flux" (with bins: "flux_bin<k>" and "flux" = their sum) and, from two batches on,
 * "flux_std_dev" / "flux_bin<k>_std_dev"; moves after the last end_batch are not part of it. */
int pumitally_get_tally_statistics(pumitally_engine *e, double *out_mean, double *out_std_dev, int64_t n);
/* Tally trigger: over the (bin, element) pairs with a non-zero mean, the largest std_dev / |mean|, the index
 * bin * num_elements + caller's element id where it is reached (lowest on ties), and how many pairs exceed
 * `threshold` (no pair with a non-zero mean: 0, -1, 0).  Needs n >= 2; every rank gets the same answer. */
int pumitally_get_max_relative_error(pumitally_engine *e, double threshold, double *out_max_rel,
                                     int64_t *out_index, int64_t *out_count_above);

/* test hook: processing order produced by the last binning pass (ids of flying particles
 * grouped by seed-grid cell); returns the number of entries, copies at most n of them */
int64_t pumitally_debug_order(pumitally_engine *e, int32_t *out, int64_t n);

/* test hook, needs no GPU: one stage pass of the host-pointer path (csrc/host_stage.hpp) over
 * particles [0, n) with `threads` workers.  b_dest/b_w/b_fly are the staging slots (b_dest also the
 * mirror the origins are compared against when compare != 0); out_patches receives 32-byte entries
 * {x, y, z, int32 index, int32 0}.  Returns the number of entries, or -1 if they exceed cap. */
int64_t pumitally_debug_stage(const double *origin, const double *dest, int8_t *flying,
                              const double *weights, double *b_dest, double *b_w, int8_t *b_fly,
                              int64_t n, int32_t compare, int32_t threads, void *out_patches,
                              int64_t cap);

const char *pumitally_version(void);

#ifdef __cplusplus
}
#endif
#endif /* PUMITALLY_C_H */
