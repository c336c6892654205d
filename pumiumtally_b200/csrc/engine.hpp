// Batch orchestration of the tally engine: owns the device-resident mesh
// tables, particle state, staging buffers, streams and the optional NCCL
// communicator.  Plays the role of the reference's PumiTallyImpl
// (reference: src/pumitally/PumiTallyImpl.h:154-221) minus everything Kokkos /
// pumi-pic / Omega_h.
#pragma once
#include <cstdint>
#include <functional>
#include <memory>
#include <string>
#include <utility>
#include <vector>

#include <cuda_runtime.h>

#include "host_stage.hpp"
#include "tet_mesh.hpp"
#include "walk_kernels.hpp"

namespace ptb {

struct EngineStats {
  uint64_t segments = 0, tracks = 0, relocations = 0, lost = 0, moves = 0;
  double kernel_ms = 0.0;
  double h2d_bytes = 0.0;
  uint64_t plane_fallbacks = 0;
};

class Engine {
 public:
  // Throws std::runtime_error when no CUDA device is usable: there is no CPU path.
  Engine(HostMesh &&mesh, int32_t num_particles, int device);
  ~Engine();
  Engine(const Engine &) = delete;
  Engine &operator=(const Engine &) = delete;

  int64_t num_elements() const { return mesh_.ntets; }
  int32_t num_particles() const { return n_; }
  const HostMesh &mesh() const { return mesh_; }

  // Host-pointer entry points (reference semantics; block until inputs are consumed).
  int copy_initial_position(const double *xyz, int32_t size);
  int move_to_next_location(const double *origin, const double *dest, int8_t *flying,
                            const double *weights, int32_t size);
  // Device-pointer entry points (enqueue only).
  int copy_initial_position_device(const double *d_xyz, int32_t size, cudaStream_t stream);
  int move_to_next_location_device(const double *d_origin, const double *d_dest,
                                   const int8_t *d_flying, const double *d_weights, int32_t size,
                                   cudaStream_t stream);

  // Score filter: nbins flux arrays; a binned move tallies particle i into array bins[i] (outside
  // [0, nbins): the particle flies unscored).  Resets the tally.  Before comm_init on multi-GPU runs.
  int set_score_bins(int32_t nbins);
  int32_t score_bins() const { return nbins_; }
  int move_to_next_location_binned(const double *origin, const double *dest, int8_t *flying, const double *weights,
                                   const int32_t *bins, int32_t size);
  int move_to_next_location_device_binned(const double *d_origin, const double *d_dest, const int8_t *d_flying,
                                          const double *d_weights, const int32_t *d_bins, int32_t size, cudaStream_t stream);
  int get_flux(double *out, int64_t n);
  // Device-side accessors, caller's element numbering, enqueued on `stream` (no synchronisation).
  int set_state_device(const double *d_xyz, const int32_t *d_elem, int32_t first, int32_t count, cudaStream_t stream);
  int get_state_device(double *d_xyz, int32_t *d_elem, int32_t first, int32_t count, cudaStream_t stream);
  int get_flux_device(double *d_out, cudaStream_t stream);
  int get_normalized_flux(double *out_flux, double *out_volume, int64_t n);
  int get_element_ids(int32_t *out, int64_t n);
  int get_positions(double *out, int64_t n3);
  int reset_tally();
  // Per-source normalisation of the *normalised* flux (get_normalized_flux, WriteTallyResults); the raw
  // flux is never touched.  0 = none (reference behaviour: flux / volume, PumiTallyImpl.cpp:402),
  // 1 = also divide by the number of particles (what PumiTally.h:93 documents), 2 = by `value`
  // (a total source weight the caller knows), 3 = by the total weight of the first tracks after
  // CopyInitialPosition / reset_tally (the reference's total_initial_weight, PumiTallyImpl.h:170-171).
  int set_source_normalization(int mode, double value);
  double source_normalization();  // the divisor currently in effect (1 for mode 0)
  int get_stats(EngineStats *out);
  int synchronize();
  double *flux_device_ptr() { return gather_shares() ? nullptr : flux_view(); }
  int set_option(const std::string &name, int64_t value);
  int64_t get_option(const std::string &name) const;
  void set_output_name(const std::string &s) { output_name_ = s; }
  int write_tally_results();
  int64_t debug_order(int32_t *out, int64_t n);

  // multi-GPU exchange step
  int comm_init(int rank, int nranks, const uint8_t id[128]);
  int allreduce_tally();
  // The cheaper batch-end exchange: every rank ends up with the sum over ranks of ITS share of the
  // elements only (ncclReduceScatter: half the traffic of the all-reduce); the shares are gathered
  // (ncclAllGather, collective) the first time a flux accessor or WriteTallyResults needs the whole array.
  int reduce_tally_to_owners();
  // whichever of the two comm_init measured to be quicker on this mesh (same choice on every rank)
  int exchange_tally();

  // Batch statistics (batch_stats.cu).  end_batch closes the batch: the tally since the last end_batch /
  // reset (summed over ranks through exchange_tally when a communicator exists), divided by the batch's
  // source divisor, is added to S1 and its square to S2 per (bin, element), and the tally and the first-track
  // weight start over.  Each rank keeps the sums of its share of the reduce-scatter layout only.  All three
  // calls are collective on several GPUs.
  int end_batch();
  // mean = S1 / n / volume and the standard deviation of the mean, caller's numbering; n as for get_flux
  int get_tally_statistics(double *out_mean, double *out_std_dev, int64_t n);
  // largest std_dev / |mean| over the pairs with a non-zero mean, its bin * E + caller's element id, and how
  // many pairs exceed `threshold` (no such pair: 0, -1, 0)
  int max_relative_error(double threshold, double *max_rel, int64_t *index, int64_t *count_above);

 private:
  int launch_range(const double *d_origin, const double *d_dest, const int8_t *d_flying,
                   const double *d_weights, int32_t begin, int32_t end, cudaStream_t stream,
                   bool timed);
  int move_host(const double *origin, const double *dest, int8_t *flying, const double *weights, int32_t size);
  int launch_range_into(double *d_flux, const double *d_origin, const double *d_dest, const int8_t *d_flying,
                        const double *d_weights, int32_t begin, int32_t end, cudaStream_t stream, bool timed);
  int32_t nbins_ = 1;
  size_t flux_alloc_ = 0;             // doubles allocated at d_flux_
  size_t flux_len() const { return size_t(nbins_) * size_t(mesh_.ntets); }  // reported part of d_flux_
  const int32_t *cur_bins_ = nullptr; // device array of the move being launched (binned moves only)
  int8_t *d_mask_ = nullptr;          // [N] flying flags of one bin
  int32_t *d_bins_ = nullptr;         // [N] bins of a host-pointer move
  int32_t *h_bins_ = nullptr;         // [N] pinned copy of the caller's bins on their way to the device
  cudaEvent_t ev_bins_ = nullptr, ev_bins_free_ = nullptr;
  bool host_is_pinned(const void *p) const;
  void maybe_register(const void *p, size_t bytes);
  void collect_timers(bool wait);
  void build_seed_grid();
  bool upload_compact();

  HostMesh mesh_;
  int32_t n_ = 0;
  int device_ = 0;
  bool initialized_ = false;  // is_pumipic_initialized (PumiTallyImpl.h:168)
  uint64_t moves_ = 0;        // iter_count (PumiTallyImpl.h:169)
  std::string output_name_ = "fluxresult.vtk";

  // options
  int variant_ = kVariantPersistRefill8;  // chosen in the constructor from mesh size vs L2 (choose_variant)
  int choose_variant() const;
  // Auto-tuner (only while the engine picks the kernel itself and the mesh is in the streaming regime):
  // whether processing the particles in spatial order pays depends on the particle data (it does for
  // collimated long tracks, config c4; it ties for isotropic ones), so the first four moves of every
  // kTuneEpoch alternate between the streaming kernel and the packed/sorted one, and the rest of the
  // epoch uses whichever had the lower kernel time.
  static constexpr uint64_t kTuneEpoch = 64;
  bool auto_variant_ = true, autotune_ = true;
  int tuned_variant_ = kVariantPersistRefill8;
  int move_variant_ = kVariantPersistRefill8, move_tag_ = -1;
  double explore_ms_[2] = {0.0, 0.0};
  int explore_pending_ = 0;
  bool explore_complete_ = false;
  uint64_t launches_ = 0;  // kernels launched by the move / localisation entry points
  void begin_move();
  int block_ = 128;
  bool chunk_user_set_ = false;
  int32_t chunk_ = 1 << 19;  // particles per H2D/compute pipeline stage (c2 from pageable arrays: 9.28 ms per move; 2^18: 10.0, 2^20: 9.5, 2^21: 10.9)
  // Seed grid for relocation / localisation.  The reference walks straight from the particle's old
  // position to the new one and stops at the hull if that segment leaves the mesh -- on a mesh with
  // concavities or voids even when the new position is inside.  Starting from a seed cell instead
  // reaches it, which is a different (better, but different) answer, so by default the shortcut is
  // used only when the hull is convex (seed_grid_mode_ 1); 0 = never, 2 = always.
  bool use_seed_grid_ = true;
  int seed_grid_mode_ = 1;
  int32_t max_iters_ = 0;  // crossing limit per walk; 0 = ntets + 16
  bool morton_ = true;    // binning key: Morton rank of the cell (matches the tet storage order) instead of its z-major index
  int claim_run_ = 4;     // chunks per ticket in gather mode

  // device memory
  TetRecord *d_tets_ = nullptr;
  TetLinks *d_links_ = nullptr;    // compact layout (walk_compact.cuh); null when the mesh exceeds its id ranges
  VertexRec *d_verts_ = nullptr;
  TetStart *d_starts_ = nullptr;
  double *d_flux_ = nullptr, *d_volume_ = nullptr, *d_scratch_ = nullptr;
  int norm_mode_ = 0;
  double norm_value_ = 1.0;
  double *d_initial_weight_ = nullptr;  // total weight of the first tracks of the batch
  bool initial_weight_pending_ = true;  // the next move is the batch's first
  ParticleState *d_state_ = nullptr;  // persistent position + parent element, 32 B per particle
  double *d_origin_ = nullptr, *d_dest_ = nullptr, *d_weights_ = nullptr;  // staging
  int8_t *d_flying_ = nullptr;
  DeviceStats *d_stats_ = nullptr;
  unsigned int *d_tickets_ = nullptr;  // ring of chunk counters for the persistent kernel
  unsigned ticket_next_ = 0;
  SeedGrid grid_{};              // relocation seed grid (grid_.cell_tet lives in d_grid_)
  int32_t *d_grid_ = nullptr;
  int32_t *d_orig_of_internal_ = nullptr, *d_internal_of_orig_ = nullptr;  // element renumbering maps (device accessors)
  int ensure_element_maps();
  int32_t *d_cell_rank_ = nullptr;
  // spatial binning of the flying particles (gather-mode kernels)
  int32_t *d_pcell_ = nullptr, *d_order_ = nullptr;
  PackedRow *d_rows_ = nullptr;  // packed variant: one 64-byte row per flying particle, allocated at first use
  unsigned int *last_work_count_ = nullptr;
  unsigned int *d_cell_count_ = nullptr, *d_cell_sums_ = nullptr, *d_work_count_ = nullptr;

  cudaStream_t compute_ = nullptr, copy_ = nullptr;
  cudaStream_t last_stream_ = nullptr;  // stream of the previous kernel launch that touched the particle state
  bool last_stream_set_ = false;
  cudaEvent_t ev_order_ = nullptr;
  struct TimerPair { cudaEvent_t a, b; int tag; };  // tag: auto-tuner slot the time belongs to, -1 = none
  std::vector<TimerPair> timers_free_, timers_busy_;
  std::vector<cudaEvent_t> chunk_events_;
  // caller buffers pinned with cudaHostRegister (option "register_host"): base -> bytes
  std::vector<std::pair<const void *, size_t>> registered_;
  bool register_host_ = false;
  double kernel_ms_ = 0.0, h2d_bytes_ = 0.0;

  // Host-pointer path, staged (host_stage.hpp): pinned per-particle slots for dest / weight / flying
  // that are both the DMA source of a move and the mirror the next move's origins are compared
  // against; only origins that changed travel, as a patch list applied to the device's copy of the
  // previous destinations.  Invariant between moves (mirror_valid_): h_dest_ == the device array
  // d_dest_, bit for bit.
  int host_path_ = 2;                 // 2 automatic (default), 1 staged, 0 direct copies from the caller's arrays
  uint64_t host_moves_ = 0;           // host-pointer moves so far (schedule of the staged-vs-direct probe)
  double span_ms_[2] = {0.0, 0.0};    // upload span per path: [0] staged, [1] direct
  int span_n_[2] = {0, 0};
  int span_tag_ = -1;                 // path of the move whose span has not been collected yet
  int span_choice_ = -1;              // this epoch's decision: 0 staged, 1 direct, -1 still probing
  void collect_upload_span();
  int mark_move_done();
  cudaEvent_t ev_done_ = nullptr;     // after the last kernel of the latest host move
  int host_threads_ = 0;              // 0 = default_host_threads() - 1
  std::unique_ptr<HostStager> stager_;  // worker pool + per-chunk stage pass
  void *stage_base_ = nullptr;
  double *h_dest_ = nullptr, *h_w_ = nullptr;
  int8_t *h_fly_ = nullptr;
  bool stage_ready_ = false, stage_failed_ = false, stage_registered_ = false;
  bool mirror_valid_ = false;
  int32_t staged_chunk_ = 0;          // chunking of the last staged move (its chunk_events_ are still meaningful)
  int staged_chunks_ = 0;
  PatchEntry *h_patch_ = nullptr;     // pinned ring of kPatchSlots chunk-sized lists
  PatchEntry *d_patch_ = nullptr;     // one list per chunk of a move
  size_t patch_cap_ = 0;              // entries per chunk
  int patch_chunks_ = 0;              // lists d_patch_ has room for
  double stage_host_s_ = 0.0, stage_sent_bytes_ = 0.0;
  cudaEvent_t ev_copy0_ = nullptr, ev_copy1_ = nullptr;  // span of the last staged move's uploads
  int pool_node_ = -1;
  int ensure_stage_buffers(const void *caller_mem, size_t caller_bytes);
  void follow_caller_memory(const void *p, size_t bytes);
  int ensure_patch_buffers(int nchunks);
  int move_direct(const double *origin, const double *dest, int8_t *flying, const double *weights, int nchunks);

  // NCCL (resolved with dlopen at comm_init time)
  void *nccl_comm_ = nullptr;
  int rank_ = 0, nranks_ = 1;
  // Result of the last batch-end exchange.  This rank's own tally keeps accumulating in d_flux_
  // across moves (reference semantics: raw flux summed over all moves); the exchange writes the
  // sum over ranks here, so it can be repeated after every batch without counting earlier batches
  // twice.  The accessors return this array until the next move or reset changes the local tally.
  double *d_flux_global_ = nullptr;
  bool flux_global_valid_ = false;
  int exchange_choice_ = 0;           // 0 all-reduce, 1 reduce-scatter to owners
  double exchange_ms_[2] = {0, 0};    // comm_init's measurement of both (mean over ranks)
  bool flux_owned_only_ = false;  // d_flux_global_ holds only this rank's share (after reduce_tally_to_owners)
  size_t share_ = 0;              // elements per rank in the scattered layout = ceil(E / nranks)
  int gather_shares();
  double *flux_view() { return flux_global_valid_ ? d_flux_global_ : d_flux_; }
  double allreduce_ms_ = 0.0;  // device time of the last exchange

  // batch statistics: running sums over the ended batches of this rank's share of the bin-major tally
  // (entries [stats_offset(), stats_offset() + stats_count()) of it), allocated at the first end_batch
  uint64_t batches_ = 0;
  double *d_s1_ = nullptr, *d_s2_ = nullptr;
  double *d_batch_small_ = nullptr;  // trigger partials and records, the divisor sum
  size_t stats_len() const { return nccl_comm_ ? share_ : flux_len(); }
  size_t stats_offset() const { return nccl_comm_ ? size_t(rank_) * share_ : 0; }
  size_t stats_count() const;
  int ensure_batch_buffers();
  void release_batch_buffers();
  int batch_divisor(double *out);
  cudaEvent_t ev_ar0_ = nullptr, ev_ar1_ = nullptr;
};

// NCCL entry points resolved with dlopen at run time (nccl_dl.cpp)
int nccl_get_unique_id(uint8_t out[128]);
int nccl_comm_init_rank(void **comm, int nranks, const uint8_t id[128], int rank);
int nccl_allreduce_sum_f64(void *comm, const double *send, double *recv, size_t count, cudaStream_t stream);
int nccl_reduce_scatter_sum_f64(void *comm, const double *send, double *recv, size_t count, cudaStream_t stream);
int nccl_all_gather_f64(void *comm, const double *send, double *recv, size_t count, cudaStream_t stream);
void nccl_comm_destroy(void *comm);

}  // namespace ptb
