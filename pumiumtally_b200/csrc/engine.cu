// Engine: device state + batch orchestration (see engine.hpp).
#include "engine.hpp"

#include <sys/mman.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <climits>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <stdexcept>

#include "batch_stats.cuh"
#include "host_stage.hpp"
#include "seed_grid.hpp"
#include "vtk_writer.hpp"

namespace ptb {

namespace {

#define PTB_CUDA_OK(expr)                                                                  \
  do {                                                                                     \
    cudaError_t _e = (expr);                                                               \
    if (_e != cudaSuccess) {                                                               \
      fprintf(stderr, "[pumitally] CUDA error %s at %s:%d: %s\n", cudaGetErrorName(_e),    \
              __FILE__, __LINE__, cudaGetErrorString(_e));                                 \
      return 1;                                                                            \
    }                                                                                      \
  } while (0)

void cuda_or_throw(cudaError_t e, const char *what) {
  if (e != cudaSuccess)
    throw std::runtime_error(std::string("[pumitally] ") + what + ": " + cudaGetErrorString(e) +
                             " (this library has no CPU fallback; a CUDA device is required)");
}

constexpr unsigned kTicketRing = 256;
constexpr size_t kFluxPad = 1024;  // most ranks a communicator may have (padding of the flux arrays)

template <typename T>
void dev_alloc(T **p, size_t count, const char *what) {
  cuda_or_throw(cudaMalloc(reinterpret_cast<void **>(p), std::max<size_t>(count, 1) * sizeof(T)), what);
}

}  // namespace

Engine::Engine(HostMesh &&mesh, int32_t num_particles, int device)
    : mesh_(std::move(mesh)), n_(num_particles) {
  if (n_ < 0) throw std::runtime_error("[pumitally] num_particles must be >= 0");
  int ndev = 0;
  cuda_or_throw(cudaGetDeviceCount(&ndev), "cudaGetDeviceCount");
  if (ndev <= 0) cuda_or_throw(cudaErrorNoDevice, "no CUDA device");
  if (device >= 0) {
    cuda_or_throw(cudaSetDevice(device), "cudaSetDevice");
    device_ = device;
  } else {
    cuda_or_throw(cudaGetDevice(&device_), "cudaGetDevice");
  }
  cuda_or_throw(cudaStreamCreateWithFlags(&compute_, cudaStreamNonBlocking), "stream");
  cuda_or_throw(cudaStreamCreateWithFlags(&copy_, cudaStreamNonBlocking), "stream");

  const size_t E = size_t(mesh_.ntets), N = size_t(n_);
  dev_alloc(&d_tets_, E, "tet records");
  flux_alloc_ = E + kFluxPad;
  dev_alloc(&d_flux_, E + kFluxPad, "flux");  // padded: the reduce-scatter exchange sends nranks equal shares
  dev_alloc(&d_volume_, E, "volume");
  dev_alloc(&d_scratch_, E, "scratch");
  dev_alloc(&d_state_, N, "particle state");
  // staging buffers (PumiTallyImpl.cpp:36-41; origin and dest get their own so one
  // upload per array suffices instead of re-using one position buffer twice)
  dev_alloc(&d_origin_, 3 * N, "origin staging");
  dev_alloc(&d_dest_, 3 * N, "dest staging");
  dev_alloc(&d_weights_, N, "weights staging");
  dev_alloc(&d_flying_, N, "flying staging");
  dev_alloc(&d_stats_, 1, "stats");
  dev_alloc(&d_initial_weight_, 1, "initial weight");
  cuda_or_throw(cudaMemset(d_initial_weight_, 0, sizeof(double)), "memset");
  dev_alloc(&d_tickets_, kTicketRing, "tickets");
  dev_alloc(&d_pcell_, N, "particle cells");
  dev_alloc(&d_order_, N, "processing order");
  dev_alloc(&d_work_count_, kTicketRing, "work counts");

  cuda_or_throw(cudaMemcpy(d_tets_, mesh_.records.data(), E * sizeof(TetRecord), cudaMemcpyHostToDevice), "upload tets");
  cuda_or_throw(cudaMemcpy(d_volume_, mesh_.volume.data(), E * sizeof(double), cudaMemcpyHostToDevice), "upload volume");
  cuda_or_throw(cudaMemset(d_flux_, 0, (E + kFluxPad) * sizeof(double)), "memset");
  cuda_or_throw(cudaMemset(d_stats_, 0, sizeof(DeviceStats)), "memset");
  // InitializeParticlesInElement0 (PumiTallyImpl.cpp:492-528)
  cuda_or_throw(launch_init_particles(d_state_, n_, mesh_.centroid0[0], mesh_.centroid0[1],
                                      mesh_.centroid0[2], mesh_.start_elem, compute_), "init particles");
  cuda_or_throw(cudaStreamSynchronize(compute_), "init sync");
  build_seed_grid();
  use_seed_grid_ = mesh_.hull_convex;  // seed_grid_mode_ 1: only where it is equivalent to the reference's walk
  if (!mesh_.hull_convex)
    printf("[INFO] pumitally-b200: the mesh hull is not convex: relocation walks go the reference's way (no seed-grid "
           "shortcut; option seed_grid=2 forces it)\n");
  variant_ = choose_variant();
  if (const char *env = std::getenv("PUMITALLY_REGISTER_HOST")) register_host_ = std::atoi(env) != 0;
  // the packed records are only needed on the device from here on
  std::vector<TetRecord>().swap(mesh_.records);
  printf("[INFO] pumitally-b200: %lld elements, %d particles on CUDA device %d\n",
         (long long)mesh_.ntets, n_, device_);
}

// Compact layout: TetLinks (32 B per tet) + vertices (32 B each) are what the edge-function walk
// reads per crossing; TetStart lines (128 B per tet) are read once per ray.  Built and uploaded the
// first time one of the edge-walk variants is selected (the default kernels never touch it).
bool Engine::upload_compact() {
#ifndef PTB_EXPERIMENTS
  return false;  // the edge-walk variants are not part of this library
#endif
  if (d_links_) return true;
  std::string err;
  if (!mesh_.build_compact(&err)) {
    printf("[INFO] pumitally-b200: compact layout not built (%s); plane records only\n", err.c_str());
    return false;
  }
  const size_t E = size_t(mesh_.ntets), V = size_t(mesh_.nverts);
  std::vector<TetLinks> links(E);
  for (size_t e = 0; e < E; ++e) links[e] = mesh_.starts[e].links;
  dev_alloc(&d_links_, E, "tet links");
  dev_alloc(&d_verts_, V, "vertices");
  dev_alloc(&d_starts_, E, "tet start lines");
  cuda_or_throw(cudaMemcpy(d_links_, links.data(), E * sizeof(TetLinks), cudaMemcpyHostToDevice), "upload links");
  cuda_or_throw(cudaMemcpy(d_verts_, mesh_.cverts.data(), V * sizeof(VertexRec), cudaMemcpyHostToDevice), "upload vertices");
  cuda_or_throw(cudaMemcpy(d_starts_, mesh_.starts.data(), E * sizeof(TetStart), cudaMemcpyHostToDevice), "upload start lines");
  std::vector<TetStart>().swap(mesh_.starts);
  std::vector<VertexRec>().swap(mesh_.cverts);
  return true;
}

Engine::~Engine() {
  cudaSetDevice(device_);
  cudaDeviceSynchronize();
  if (nccl_comm_) nccl_comm_destroy(nccl_comm_);
  cudaFree(d_flux_global_);
  release_batch_buffers();
  if (ev_order_) cudaEventDestroy(ev_order_);
  if (ev_done_) cudaEventDestroy(ev_done_);
  if (ev_bins_) cudaEventDestroy(ev_bins_);
  if (ev_bins_free_) cudaEventDestroy(ev_bins_free_);
  cudaFree(d_mask_);
  cudaFree(d_bins_);
  if (h_bins_) cudaFreeHost(h_bins_);
  if (ev_copy0_) cudaEventDestroy(ev_copy0_);
  if (ev_copy1_) cudaEventDestroy(ev_copy1_);
  if (ev_ar0_) cudaEventDestroy(ev_ar0_);
  if (ev_ar1_) cudaEventDestroy(ev_ar1_);
  for (auto &r : registered_) cudaHostUnregister(const_cast<void *>(r.first));
  for (auto &t : timers_free_) { cudaEventDestroy(t.a); cudaEventDestroy(t.b); }
  for (auto &t : timers_busy_) { cudaEventDestroy(t.a); cudaEventDestroy(t.b); }
  for (auto &e : chunk_events_) cudaEventDestroy(e);
  stager_.reset();
  if (stage_base_) {
    if (stage_registered_) { cudaHostUnregister(stage_base_); free(stage_base_); }
    else cudaFreeHost(stage_base_);
  }
  cudaFree(d_rows_);
  if (h_patch_) cudaFreeHost(h_patch_);
  cudaFree(d_patch_);
  cudaFree(d_links_); cudaFree(d_verts_); cudaFree(d_starts_);
  cudaFree(d_tets_); cudaFree(d_flux_); cudaFree(d_volume_); cudaFree(d_scratch_);
  cudaFree(d_state_);
  cudaFree(d_origin_); cudaFree(d_dest_); cudaFree(d_weights_); cudaFree(d_flying_);
  cudaFree(d_stats_);
  cudaFree(d_initial_weight_);
  cudaFree(d_tickets_);
  cudaFree(d_grid_);
  cudaFree(d_orig_of_internal_); cudaFree(d_internal_of_orig_);
  cudaFree(d_cell_rank_);
  cudaFree(d_pcell_); cudaFree(d_order_); cudaFree(d_cell_count_); cudaFree(d_cell_sums_);
  cudaFree(d_work_count_);
  if (compute_) cudaStreamDestroy(compute_);
  if (copy_) cudaStreamDestroy(copy_);
}

// Localise the seed point of every grid cell with the walk kernel itself (from the centroid of
// element 0, like any particle) and keep the tet for cells whose seed point lies in the mesh.
void Engine::build_seed_grid() {
  grid_ = choose_seed_grid(mesh_);
  const int32_t ncell = grid_.nx * grid_.ny * grid_.nz;
  double *xyz = nullptr;
  ParticleState *ts = nullptr;
  dev_alloc(&d_grid_, size_t(ncell), "seed grid");
  dev_alloc(&xyz, 3 * size_t(ncell), "seed points");
  dev_alloc(&ts, size_t(ncell), "seed tmp");
  cuda_or_throw(launch_seed_points(grid_, xyz, compute_), "seed points");
  cuda_or_throw(launch_init_particles(ts, ncell, mesh_.centroid0[0], mesh_.centroid0[1],
                                      mesh_.centroid0[2], mesh_.start_elem, compute_), "seed init");
  WalkParams p{};
  p.tets = d_tets_;
  p.flux = d_flux_;
  p.state = ts;
  p.origin = xyz;
  p.begin = 0;
  p.end = ncell;
  p.max_iters = int32_t(std::min<int64_t>(mesh_.ntets + 16, INT_MAX));
  p.bulk_ok = 1;
  p.work_counter = d_tickets_;
  p.stats = d_stats_;
  p.cx = mesh_.center[0]; p.cy = mesh_.center[1]; p.cz = mesh_.center[2];
  cuda_or_throw(launch_walk(p, kVariantPersistRefill8, 128, compute_), "seed walk");
  cuda_or_throw(launch_seed_finalize(xyz, ts, d_grid_, ncell, compute_), "seed finalize");
  cuda_or_throw(cudaStreamSynchronize(compute_), "seed sync");
  cuda_or_throw(cudaMemset(d_stats_, 0, sizeof(DeviceStats)), "memset");
  cudaFree(xyz); cudaFree(ts);
  grid_.cell_tet = d_grid_;
  {
    const std::vector<int32_t> rank = morton_cell_ranks(grid_);
    dev_alloc(&d_cell_rank_, size_t(ncell), "cell ranks");
    cuda_or_throw(cudaMemcpy(d_cell_rank_, rank.data(), size_t(ncell) * sizeof(int32_t), cudaMemcpyHostToDevice), "upload cell ranks");
    grid_.cell_rank = d_cell_rank_;
  }
  dev_alloc(&d_cell_count_, size_t(ncell), "cell histogram");
  dev_alloc(&d_cell_sums_, size_t(ncell) / 1024 + 2, "cell block sums");
}

void Engine::collect_timers(bool wait) {
  for (size_t k = 0; k < timers_busy_.size();) {
    TimerPair t = timers_busy_[k];
    if (wait) cudaEventSynchronize(t.b);
    if (cudaEventQuery(t.b) == cudaSuccess) {
      float ms = 0.f;
      if (cudaEventElapsedTime(&ms, t.a, t.b) == cudaSuccess) kernel_ms_ += ms;
      if (t.tag >= 0) {
        explore_ms_[t.tag] += ms;
        if (--explore_pending_ == 0 && explore_complete_) {  // all four exploration moves measured
          // the streaming kernel keeps the job unless sorting buys more than 3 %
          tuned_variant_ = (explore_ms_[1] > 0.0 && explore_ms_[1] < 0.97 * explore_ms_[0]) ? kVariantPacked : kVariantPersistRefill8;
          explore_complete_ = false;
        }
      }
      timers_free_.push_back(t);
      timers_busy_[k] = timers_busy_.back();
      timers_busy_.pop_back();
    } else {
      ++k;
    }
  }
}

// Picks the kernel for the move that is about to be launched (see the auto-tuner note in engine.hpp).
void Engine::begin_move() {
  collect_timers(false);
  move_variant_ = variant_;
  move_tag_ = -1;
  if (!auto_variant_ || !autotune_ || variant_ != kVariantPersistRefill8) return;
  // sorting costs per particle, walking per crossing: with thousands of particles per tet (config c3) the
  // sorted variant cannot win and two exploration moves would cost more than an epoch can pay back
  if (int64_t(n_) > 16 * mesh_.ntets) return;
  // exploration moves 1..4 of every epoch in the order streaming, packed, packed, streaming (move 0 of a
  // run is atypical: nothing has been re-sourced yet); decision when all four have been timed
  const uint64_t k = moves_ % kTuneEpoch;
  if (k >= 1 && k <= 4) {
    if (k == 1) { explore_ms_[0] = explore_ms_[1] = 0.0; explore_complete_ = false; }
    move_tag_ = (k == 2 || k == 3) ? 1 : 0;
    move_variant_ = move_tag_ ? kVariantPacked : kVariantPersistRefill8;
  } else {
    if (k == 5) {
      explore_complete_ = true;  // every exploration launch has been issued
      // a caller that queues moves back to back has not let the four timed moves finish yet: wait for
      // them once per epoch (a bubble of at most one move) rather than decide an epoch late
      for (auto &t : timers_busy_)
        if (t.tag >= 0) cudaEventSynchronize(t.b);
      collect_timers(false);
      if (explore_complete_ && explore_pending_ == 0) {
        tuned_variant_ = (explore_ms_[1] > 0.0 && explore_ms_[1] < 0.97 * explore_ms_[0]) ? kVariantPacked : kVariantPersistRefill8;
        explore_complete_ = false;
      }
    }
    move_variant_ = tuned_variant_;
  }
}

int Engine::launch_range(const double *d_origin, const double *d_dest, const int8_t *d_flying,
                         const double *d_weights, int32_t begin, int32_t end, cudaStream_t stream,
                         bool timed) {
  if (end <= begin) return 0;
  // Particle state, binning scratch and the ticket ring are shared by every launch: work enqueued on
  // another stream than the previous launch's (a device-pointer move on the caller's stream after a
  // host-pointer move on the engine's own, or the other way round) is ordered behind it by an event.
  if (last_stream_set_ && stream != last_stream_) {
    if (!ev_order_) PTB_CUDA_OK(cudaEventCreateWithFlags(&ev_order_, cudaEventDisableTiming));
    PTB_CUDA_OK(cudaEventRecord(ev_order_, last_stream_));
    PTB_CUDA_OK(cudaStreamWaitEvent(stream, ev_order_, 0));
  }
  last_stream_ = stream;
  last_stream_set_ = true;
  if (d_dest) flux_global_valid_ = flux_owned_only_ = false;  // the local tally moves on; the last exchange no longer describes it
  if (!(cur_bins_ && d_dest)) return launch_range_into(d_flux_, d_origin, d_dest, d_flying, d_weights, begin, end, stream, timed);
  // Score filter: particles are independent and a particle that does not fly is not touched, so the range
  // is walked once per bin with the flying flags masked down to that bin's particles and the tally pointed
  // at that bin's flux array -- the walk kernels themselves are the unfiltered ones.  One more pass (array
  // nbins_, never reported) flies the particles whose bin is outside [0, nbins_): they move, unscored.
  // The streaming kernel pays for every particle of the range in every pass, flying or not (measured on c2:
  // 2.7 ms unfiltered, 5.5 ms with 4 bins, 10.3 ms with 8); the packed kernel's sort pass keeps only the flying
  // ones, so its passes cost what their members cost.  Unless the caller has fixed the kernel, binned moves use it.
  const int saved_variant = move_variant_, saved_tag = move_tag_;
  if (auto_variant_ && d_weights) {
    move_variant_ = kVariantPacked;
    move_tag_ = -1;  // not one of the auto-tuner's exploration moves
  }
  int rc = 0;
  for (int32_t b = 0; b <= nbins_ && !rc; ++b) {
    if (launch_bin_mask(d_flying, cur_bins_, b, nbins_, d_mask_, begin, end, stream) != cudaSuccess) { rc = 1; break; }
    ++launches_;
    rc = launch_range_into(d_flux_ + size_t(b) * size_t(mesh_.ntets), d_origin, d_dest, d_mask_, d_weights, begin, end, stream, timed);
  }
  move_variant_ = saved_variant;
  move_tag_ = saved_tag;
  return rc;
}

int Engine::launch_range_into(double *d_flux, const double *d_origin, const double *d_dest, const int8_t *d_flying,
                              const double *d_weights, int32_t begin, int32_t end, cudaStream_t stream, bool timed) {
  if (d_dest && d_weights && initial_weight_pending_)  // first tracks of the batch: their total weight
    PTB_CUDA_OK(launch_sum_flying_weights(d_flying, d_weights, begin, end, d_initial_weight_, stream));
  WalkParams p{};
  p.tets = d_tets_;
  p.links = d_links_;
  p.verts = d_verts_;
  p.starts = d_starts_;
  p.flux = d_flux;
  p.state = d_state_;
  p.origin = d_origin;
  p.dest = d_dest;
  p.flying = d_flying;
  p.weights = d_weights;
  p.begin = begin;
  p.end = end;
  p.max_iters = max_iters_ > 0 ? max_iters_ : int32_t(std::min<int64_t>(mesh_.ntets + 16, INT_MAX));
  p.stats = d_stats_;
  p.grid = grid_;
  p.cx = mesh_.center[0]; p.cy = mesh_.center[1]; p.cz = mesh_.center[2];
  if (!use_seed_grid_) p.grid.cell_tet = nullptr;
  p.work_counter = d_tickets_ + (ticket_next_++ % kTicketRing);
  auto aligned16 = [](const void *q) { return (reinterpret_cast<uintptr_t>(q) & 15u) == 0; };
  p.bulk_ok = (begin % 16 == 0) && aligned16(d_origin) && aligned16(d_dest) && aligned16(d_flying) &&
              aligned16(d_weights);
  TimerPair t{};
  t.tag = -1;
  if (timed) {
    if (timers_free_.empty()) {
      PTB_CUDA_OK(cudaEventCreate(&t.a));
      PTB_CUDA_OK(cudaEventCreate(&t.b));
    } else {
      t = timers_free_.back();
      timers_free_.pop_back();
    }
    t.tag = move_tag_;
    if (t.tag >= 0) ++explore_pending_;
    PTB_CUDA_OK(cudaEventRecord(t.a, stream));
  }
  int variant = move_variant_;
  const bool packed = variant_is_packed(variant);
  if (packed && !(d_dest && d_weights)) variant = kVariantPersistRefill8;  // localisation
  bool use_packed = packed && variant == move_variant_;
  if (use_packed && !d_rows_ &&
      cudaMalloc(reinterpret_cast<void **>(&d_rows_), std::max<size_t>(size_t(n_), 1) * sizeof(PackedRow)) != cudaSuccess) {
    cudaGetLastError();
    d_rows_ = nullptr;
    if (auto_variant_) {  // the auto-tuner wanted to try it: carry on with the streaming kernel for good
      autotune_ = false;
      tuned_variant_ = variant = move_variant_ = kVariantPersistRefill8;
      use_packed = false;
    } else {
      fprintf(stderr, "[pumitally] ERROR: no device memory for the packed particle rows\n");
      return 1;
    }
  }
  if (use_packed) {
    // counting sort by seed-grid cell, the scatter pass writing one 64-byte row per flying particle
    unsigned int *wc = d_work_count_ + (ticket_next_ % kTicketRing);
    SeedGrid bin_grid = grid_;
    if (!morton_) bin_grid.cell_rank = nullptr;
    PTB_CUDA_OK(launch_bin_pack_particles(bin_grid, d_origin, d_dest, d_weights, d_flying, d_state_, begin, end,
                                          d_pcell_, d_cell_count_, d_cell_sums_, d_rows_ + begin, wc, stream));
    p.rows = d_rows_ + begin;
    p.work_count = wc;
    last_work_count_ = wc;
    p.flying = nullptr;  // only flying particles have rows
    launches_ += 5;  // count, 3-kernel scan, pack
  }
  if (variant_is_gather(variant)) {
    // counting sort of the range's flying particles by seed-grid cell of their origin
    unsigned int *wc = d_work_count_ + (ticket_next_ % kTicketRing);
    SeedGrid bin_grid = grid_;
    if (!morton_) bin_grid.cell_rank = nullptr;
    p.claim_run = claim_run_;
    PTB_CUDA_OK(launch_bin_particles(bin_grid, d_origin, d_state_, d_flying, begin, end, d_pcell_, d_cell_count_,
                                     d_cell_sums_, d_order_ + begin, wc, stream));
    p.order = d_order_ + begin;
    p.work_count = wc;
    last_work_count_ = wc;
    launches_ += 5;  // count, 3-kernel scan, scatter
    p.flying = nullptr;  // order[] holds flying particles only
  }
  PTB_CUDA_OK(launch_walk(p, variant, block_, stream));
  ++launches_;
  if (timed) {
    PTB_CUDA_OK(cudaEventRecord(t.b, stream));
    timers_busy_.push_back(t);
  }
  return 0;
}

// OpenMC hands over ordinary (pageable) std::vector storage and reuses the same buffers for every
// call.  Pageable cudaMemcpyAsync is staged by the driver at a fraction of the PCIe rate, so with
// option register_host=1 (or PUMITALLY_REGISTER_HOST=1) each new caller buffer is page-locked once
// with cudaHostRegister and stays registered until the engine is destroyed.  Off by default: the
// caller must then keep those buffers alive (or at least not free them) for the engine's lifetime.
void Engine::maybe_register(const void *p, size_t bytes) {
  if (!register_host_ || !p || bytes == 0 || host_is_pinned(p)) return;
  for (auto &r : registered_)
    if (r.first == p && r.second >= bytes) return;
  if (cudaHostRegister(const_cast<void *>(p), bytes, cudaHostRegisterDefault) == cudaSuccess)
    registered_.emplace_back(p, bytes);
  else
    cudaGetLastError();  // overlapping/foreign registration: fall back to the pageable path
}

bool Engine::host_is_pinned(const void *p) const {
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
    cudaGetLastError();
    return false;
  }
  return a.type == cudaMemoryTypeHost;
}

// CopyInitialPositionToBuffer + MoveToInitialLocation (PumiTallyImpl.cpp:54-64, 195-221)
int Engine::copy_initial_position(const double *xyz, int32_t size) {
  if (int64_t(size) != 3 * int64_t(n_)) {
    fprintf(stderr, "[pumitally] ERROR: CopyInitialPosition size %d != 3 * num_particles (%d)\n", size, n_);
    return 1;
  }
  if (initialized_) {
    fprintf(stderr, "[pumitally] ERROR: CopyInitialPosition may only be called once\n");
    return 1;
  }
  PTB_CUDA_OK(cudaSetDevice(device_));
  // Through the staging slots when they can be had: the pool copies xyz into the pinned dest slots
  // (pageable cudaMemcpy runs at a fifth of the PCIe rate) and the device copy goes to d_dest_, so
  // that "pinned dest slots == device dest array == where every particle is" already holds for the
  // first move and its origins need not travel either.
  const double *src = xyz;
  double *d_xyz = d_origin_;
  if (host_path_ != 0 && n_ > 0 && ensure_stage_buffers(xyz, size_t(size) * sizeof(double)) == 0) {
    HostPool *pool_ = &stager_->pool();
    const int T = pool_->size();
    const int64_t total = int64_t(size);
    pool_->run([&](int t) {
      const int64_t lo = (total * t / T) & ~int64_t(7), hi = t == T - 1 ? total : (total * (t + 1) / T) & ~int64_t(7);
      std::memcpy(h_dest_ + lo, xyz + lo, size_t(hi - lo) * sizeof(double));
    });
    src = h_dest_;
    d_xyz = d_dest_;
    mirror_valid_ = true;
  }
  PTB_CUDA_OK(cudaMemcpyAsync(d_xyz, src, size_t(size) * sizeof(double), cudaMemcpyHostToDevice, compute_));
  h2d_bytes_ += double(size) * sizeof(double);
  move_variant_ = variant_;
  move_tag_ = -1;
  if (launch_range(d_xyz, nullptr, nullptr, nullptr, 0, n_, compute_, true)) return 1;
  PTB_CUDA_OK(cudaStreamSynchronize(compute_));
  initialized_ = true;
  return 0;
}

int Engine::copy_initial_position_device(const double *d_xyz, int32_t size, cudaStream_t stream) {
  if (int64_t(size) != 3 * int64_t(n_) || initialized_) {
    fprintf(stderr, "[pumitally] ERROR: CopyInitialPosition: bad size or called twice\n");
    return 1;
  }
  PTB_CUDA_OK(cudaSetDevice(device_));
  move_variant_ = variant_;
  move_tag_ = -1;
  if (launch_range(d_xyz, nullptr, nullptr, nullptr, 0, n_, stream, true)) return 1;
  initialized_ = true;
  return 0;
}

constexpr int kPatchSlots = 4;             // pinned patch lists in flight
constexpr double kPatchMaxFraction = 0.4;  // above this share of changed origins a chunk is sent whole

// Pinned staging ("bounce") buffers of the host-pointer path, allocated at the first host call:
// one slot per particle for dest, weight and flying.  They are the DMA source of every move AND the
// mirror the next move's origins are compared against (host_stage.hpp).  Ordinary page-aligned
// memory, first touched by the pool's workers (which run on the GPU's NUMA node) and then
// page-locked with cudaHostRegister -- an order of magnitude faster than cudaHostAlloc for
// hundreds of MB; cudaHostAlloc is the fallback.
// The workers follow the caller's memory: if the arrays of this call live on another NUMA node than
// the one the pool runs on, the workers move there (a few microseconds, once per change).
void Engine::follow_caller_memory(const void *p, size_t bytes) {
  if (!stager_) return;
  const int node = numa_node_of(p, bytes);
  if (node < 0 || node == pool_node_) return;
  const std::vector<int> cpus = numa_node_cpus(node);
  if (cpus.empty()) return;
  stager_->pool().repin(cpus);
  pool_node_ = node;
}

int Engine::ensure_stage_buffers(const void *caller_mem, size_t caller_bytes) {
  if (stage_ready_) return 0;
  if (stage_failed_) return 1;
  const size_t N = std::max<size_t>(size_t(n_), 1);
  if (!stager_) {
    // workers (and, by first touch, the staging slots) on the NUMA node of the caller's arrays; when
    // that cannot be determined, on the GPU's node
    std::vector<int> cpus;
    pool_node_ = numa_node_of(caller_mem, caller_bytes);
    if (pool_node_ >= 0) cpus = numa_node_cpus(pool_node_);
    if (cpus.empty()) {
      char bus[64] = {0};
      pool_node_ = -1;
      if (cudaDeviceGetPCIBusId(bus, sizeof(bus), device_) == cudaSuccess) cpus = gpu_local_cpus(bus);
      else cudaGetLastError();
    }
    // one of the CPUs the quota allows is left to the calling thread, which enqueues copies and kernels
    stager_.reset(new HostStager(host_threads_ > 0 ? host_threads_ : std::max(1, default_host_threads() - 1), cpus));
  }
  HostPool *pool_ = &stager_->pool();
  const size_t bytes_dest = (3 * N * sizeof(double) + 4095) & ~size_t(4095);
  const size_t bytes_w = (N * sizeof(double) + 4095) & ~size_t(4095);
  const size_t bytes_fly = (N + 4095) & ~size_t(4095);
  const size_t total = bytes_dest + bytes_w + bytes_fly;
  void *base = nullptr;
  if (posix_memalign(&base, size_t(2) << 20, total) == 0) {
    madvise(base, total, MADV_HUGEPAGE);  // 2 MB pages where the kernel offers them: three streams of TLB misses less
    const int T = pool_->size();
    pool_->run([&](int t) {  // first touch on the workers' NUMA node
      const size_t lo = (total * size_t(t) / size_t(T)) & ~size_t(4095);
      const size_t hi = t == T - 1 ? total : (total * size_t(t + 1) / size_t(T)) & ~size_t(4095);
      std::memset(static_cast<char *>(base) + lo, 0, hi - lo);
    });
    if (cudaHostRegister(base, total, cudaHostRegisterDefault) == cudaSuccess) {
      stage_registered_ = true;
    } else {
      cudaGetLastError();
      free(base);
      base = nullptr;
    }
  }
  if (!base) {
    if (cudaHostAlloc(&base, total, cudaHostAllocDefault) != cudaSuccess) {
      cudaGetLastError();
      stage_failed_ = true;  // the direct path (plain copies from the caller's memory) still works
      fprintf(stderr, "[pumitally] WARNING: no pinned host memory for the staging buffers (%zu MB); "
                      "uploads fall back to direct copies from the caller's arrays\n", total >> 20);
      return 1;
    }
    stage_registered_ = false;
  }
  stage_base_ = base;
  h_dest_ = static_cast<double *>(base);
  h_w_ = reinterpret_cast<double *>(static_cast<char *>(base) + bytes_dest);
  h_fly_ = reinterpret_cast<int8_t *>(static_cast<char *>(base) + bytes_dest + bytes_w);
  stager_->set_buffers(h_dest_, h_w_, h_fly_);
  stage_ready_ = true;
  return 0;
}

int Engine::ensure_patch_buffers(int nchunks) {
  size_t cap = size_t(double(std::min<int64_t>(chunk_, n_)) * kPatchMaxFraction) + 64;
  if (h_patch_ && patch_cap_ >= cap && patch_chunks_ >= nchunks) return 0;
  // (grow only, in both dimensions: moves with different stage sizes -- binned and plain -- may alternate)
  cap = std::max(cap, patch_cap_);
  nchunks = std::max(nchunks, patch_chunks_);
  PTB_CUDA_OK(cudaDeviceSynchronize());
  if (h_patch_) cudaFreeHost(h_patch_);
  if (d_patch_) cudaFree(d_patch_);
  h_patch_ = nullptr;
  d_patch_ = nullptr;
  patch_cap_ = cap;
  patch_chunks_ = nchunks;
  PTB_CUDA_OK(cudaHostAlloc(reinterpret_cast<void **>(&h_patch_), cap * kPatchSlots * sizeof(PatchEntry), cudaHostAllocDefault));
  PTB_CUDA_OK(cudaMalloc(reinterpret_cast<void **>(&d_patch_), cap * size_t(nchunks) * sizeof(PatchEntry)));
  stager_->reserve(cap);
  return 0;
}

// MoveToNextLocation (PumiTallyImpl.cpp:66-149), host pointers.
//
// Staged path (default): the particle range is cut into chunks; for each chunk the pool refills the
// pinned staging slots from the caller's arrays and finds the origins that differ from the previous
// destinations (stage_chunk), then flying + patch list + dest + weights of the chunk are enqueued on
// the copy stream and the walk kernel of the chunk behind them on the compute stream -- chunk k is
// on the wire and chunk k-1 is being walked while the pool stages chunk k+1.  The device's copy of
// the previous destinations becomes this move's origin array (buffer swap) and only the changed
// origins are patched in, so 32 B + a few patch bytes per particle cross PCIe instead of 57 B.  The
// call returns as soon as the caller's arrays have been consumed (they are in the staging buffers
// by then; reference: blocking deep_copy); copies and kernels may still be in flight.
//
// Direct path (option host_path=0, or no pinned memory to be had): plain cudaMemcpyAsync of all
// four arrays from the caller's memory, optionally page-locked first (option register_host).
int Engine::move_to_next_location(const double *origin, const double *dest, int8_t *flying,
                                  const double *weights, int32_t size) {
  if (int64_t(size) != 3 * int64_t(n_)) {
    fprintf(stderr, "[pumitally] ERROR: MoveToNextLocation size %d != 3 * num_particles (%d)\n", size, n_);
    return 1;
  }
  if (!initialized_) {
    fprintf(stderr, "[pumitally] ERROR: MoveToNextLocation before CopyInitialPosition\n");
    return 1;
  }
  PTB_CUDA_OK(cudaSetDevice(device_));
  begin_move();
  // Pipeline stage size, unless the caller set it: 512 Ki particles for the streaming kernel (shortest tail); the
  // sorted kernels pay a fixed price per launch (a scan over all seed-grid cells), so their stages are 2 Mi
  // (c5 share, 50 M particles per GPU from pageable arrays: 58.6 ms per move with 1 Mi stages, 86.5 ms with 512 Ki).
  const int32_t chunk = chunk_;
  // The auto-tuner compares kernel times; in a host move the sorted kernel it may prefer would also need the
  // larger stages, whose longer tail costs more than the kernel wins (c2 from pageable arrays: 11.1 ms against
  // 9.4 ms per move).  So a host move of more than one stage keeps the engine's base kernel and does not take
  // part in the exploration; the tuner works for device-pointer moves and single-stage host moves (c4's 1 M tracks).
  if (auto_variant_ && variant_is_packed(move_variant_) && !variant_is_packed(variant_) && n_ > chunk_) {
    move_variant_ = variant_;
    move_tag_ = -1;
  }
  if (!chunk_user_set_ && (variant_is_gather(move_variant_) || variant_is_packed(move_variant_)))
    chunk_ = std::max(chunk_, int32_t(1) << 21);
  const int rc = move_host(origin, dest, flying, weights, size);
  chunk_ = chunk;
  return rc;
}

int Engine::move_host(const double *origin, const double *dest, int8_t *flying, const double *weights, int32_t size) {
  const int nchunks = n_ ? (n_ + chunk_ - 1) / chunk_ : 0;
  while (int(chunk_events_.size()) < nchunks + 2) {
    cudaEvent_t e;
    PTB_CUDA_OK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    chunk_events_.push_back(e);
  }
  if (register_host_) {  // opt-in: page-lock the caller's arrays the first time they are seen
    maybe_register(origin, 3 * size_t(n_) * sizeof(double));
    maybe_register(dest, 3 * size_t(n_) * sizeof(double));
    maybe_register(weights, size_t(n_) * sizeof(double));
    maybe_register(flying, size_t(n_));
  }
  // host_path 2 (default): staged, except that page-locked caller arrays (which the direct path can DMA
  // at the full PCIe rate without any host work) get the faster of the two, measured: moves 2-3 of every
  // 256 go direct, the others staged until the upload spans of both are known.  Where the host is the
  // scarce resource -- several ranks sharing one socket's memory system -- direct wins; with cores and
  // bandwidth to spare, staged does (DESIGN.md section 5).
  bool want_staged = host_path_ != 0;
  int probe = -1;
  if (host_path_ == 2 && host_is_pinned(origin) && host_is_pinned(dest) && host_is_pinned(weights) && host_is_pinned(flying)) {
    collect_upload_span();
    const uint64_t k = host_moves_ % 256;
    if (k == 0) { span_ms_[0] = span_ms_[1] = 0.0; span_n_[0] = span_n_[1] = 0; span_choice_ = -1; }
    if (k >= 2 && k <= 3) {
      probe = 1;
    } else if (k <= 1 || span_n_[0] == 0 || span_n_[1] == 0) {
      probe = 0;
    } else {
      // decided once per epoch, from the probe moves only: changing paths is not free (the first staged move
      // after a direct one has no mirror and sends every origin)
      if (span_choice_ < 0) {
        span_choice_ = (span_ms_[1] / span_n_[1] < 0.9 * span_ms_[0] / span_n_[0]) ? 1 : 0;
        if (std::getenv("PUMITALLY_DEBUG_SPANS"))
          fprintf(stderr, "[pumitally] staged %.3f ms, direct %.3f ms per move -> %s\n", span_ms_[0] / span_n_[0],
                  span_ms_[1] / span_n_[1], span_choice_ ? "direct" : "staged");
      }
      probe = span_choice_;
    }
    want_staged = probe == 0;
  }
  ++host_moves_;
  span_tag_ = probe;
  const bool staged = want_staged && n_ > 0 && ensure_stage_buffers(dest, size_t(size) * sizeof(double)) == 0 &&
                      ensure_patch_buffers(nchunks) == 0;
  if (!staged) return move_direct(origin, dest, flying, weights, nchunks);
  follow_caller_memory(dest, size_t(size) * sizeof(double));

  // a chunk's staging slots may be refilled once the previous move's copies out of them are done;
  // with an unchanged chunking that is chunk_events_[k], otherwise wait for the whole copy stream
  if (staged_chunk_ != chunk_ || staged_chunks_ != nchunks) {
    PTB_CUDA_OK(cudaStreamSynchronize(copy_));
    staged_chunks_ = 0;
  }
  const bool compare = mirror_valid_;
  mirror_valid_ = false;  // until this move has gone through completely
  cudaEvent_t ev_prev_done = chunk_events_[nchunks];
  // the device staging arrays are free once the previous move's kernels have finished
  PTB_CUDA_OK(cudaEventRecord(ev_prev_done, compute_));
  PTB_CUDA_OK(cudaStreamWaitEvent(copy_, ev_prev_done, 0));
  // the previous destinations, still on the device, are this move's origins before patching
  if (compare) std::swap(d_origin_, d_dest_);
  double sent = 0.0;
  bool caller_memory_on_the_wire = false;
  const auto t_begin = std::chrono::steady_clock::now();
  auto range_of = [&](int k, int32_t &b, int32_t &e) {
    b = int32_t(int64_t(k) * chunk_);
    e = int32_t(std::min<int64_t>(n_, int64_t(b) + chunk_));
  };
  // the staging slots of chunk k may be refilled once the previous move's copies out of them are done,
  // its pinned patch slot once the copies of chunk k - kPatchSlots of this move are done
  auto start_stage = [&](int k) -> int {
    if (k < staged_chunks_) PTB_CUDA_OK(cudaEventSynchronize(chunk_events_[k]));
    if (k >= kPatchSlots) PTB_CUDA_OK(cudaEventSynchronize(chunk_events_[k - kPatchSlots]));
    int32_t b, e;
    range_of(k, b, e);
    stager_->begin(origin, dest, flying, weights, b, e, compare, h_patch_ + size_t(k % kPatchSlots) * patch_cap_);
    return 0;
  };
  if (!ev_copy0_) {
    PTB_CUDA_OK(cudaEventCreate(&ev_copy0_));
    PTB_CUDA_OK(cudaEventCreate(&ev_copy1_));
  }
  PTB_CUDA_OK(cudaEventRecord(ev_copy0_, copy_));
  if (nchunks > 0 && start_stage(0)) return 1;
  for (int k = 0; k < nchunks; ++k) {
    int32_t b, e;
    range_of(k, b, e);
    const size_t cnt = size_t(e - b);
    const int64_t npatch = stager_->end();  // chunk k is staged
    // the workers stage chunk k+1 while this thread enqueues the copies and kernels of chunk k
    if (k + 1 < nchunks && start_stage(k + 1)) return 1;
    PatchEntry *hp = h_patch_ + size_t(k % kPatchSlots) * patch_cap_, *dp = d_patch_ + size_t(k) * patch_cap_;
    PTB_CUDA_OK(cudaMemcpyAsync(d_flying_ + b, h_fly_ + b, cnt, cudaMemcpyHostToDevice, copy_));
    if (!compare || npatch < 0) {  // no usable mirror, or too many changed origins: the slice travels whole
      PTB_CUDA_OK(cudaMemcpyAsync(d_origin_ + 3 * size_t(b), origin + 3 * size_t(b), 3 * cnt * sizeof(double), cudaMemcpyHostToDevice, copy_));
      sent += 24.0 * double(cnt);
      caller_memory_on_the_wire = true;
    } else if (npatch > 0) {
      PTB_CUDA_OK(cudaMemcpyAsync(dp, hp, size_t(npatch) * sizeof(PatchEntry), cudaMemcpyHostToDevice, copy_));
      sent += double(npatch) * sizeof(PatchEntry);
    }
    PTB_CUDA_OK(cudaMemcpyAsync(d_dest_ + 3 * size_t(b), h_dest_ + 3 * size_t(b), 3 * cnt * sizeof(double), cudaMemcpyHostToDevice, copy_));
    PTB_CUDA_OK(cudaMemcpyAsync(d_weights_ + b, h_w_ + b, cnt * sizeof(double), cudaMemcpyHostToDevice, copy_));
    sent += 33.0 * double(cnt);
    PTB_CUDA_OK(cudaEventRecord(chunk_events_[k], copy_));
    PTB_CUDA_OK(cudaStreamWaitEvent(compute_, chunk_events_[k], 0));
    if (compare && npatch > 0) {
      PTB_CUDA_OK(launch_patch_origins(d_origin_, dp, int32_t(npatch), compute_));
      ++launches_;
    }
    if (launch_range(d_origin_, d_dest_, d_flying_, d_weights_, b, e, compute_, true)) return 1;
  }
  PTB_CUDA_OK(cudaEventRecord(ev_copy1_, copy_));
  if (mark_move_done()) return 1;
  // origin slices that went whole were read from the caller's own memory (asynchronously, if it is
  // pinned): they must be on the device before the caller gets its arrays back
  if (caller_memory_on_the_wire) PTB_CUDA_OK(cudaStreamSynchronize(copy_));
  stage_host_s_ = std::chrono::duration<double>(std::chrono::steady_clock::now() - t_begin).count();
  stage_sent_bytes_ = sent;
  h2d_bytes_ += sent;
  staged_chunk_ = chunk_;
  staged_chunks_ = nchunks;
  mirror_valid_ = true;
  initial_weight_pending_ = false;
  ++moves_;
  return 0;
}

// Device time the previous host move's uploads took (first copy could start -> last copy done), credited to
// the path that move used; feeds the staged-vs-direct choice for page-locked caller arrays.
void Engine::collect_upload_span() {
  if (span_tag_ < 0 || !ev_copy0_) return;
  if (span_choice_ >= 0) { span_tag_ = -1; return; }  // decided for this epoch
  float ms = 0.f;
  if (ev_done_ && cudaEventSynchronize(ev_done_) == cudaSuccess && cudaEventElapsedTime(&ms, ev_copy0_, ev_done_) == cudaSuccess) {
    span_ms_[span_tag_] += ms;
    ++span_n_[span_tag_];
    if (std::getenv("PUMITALLY_DEBUG_SPANS"))
      fprintf(stderr, "[pumitally] host move %llu: %s path, uploads + walk %.3f ms on the device\n",
              (unsigned long long)host_moves_ - 1, span_tag_ ? "direct" : "staged", ms);
  } else {
    cudaGetLastError();
  }
  span_tag_ = -1;
}

// marks the end of a host move's device work (after its last kernel): what collect_upload_span() measures up to
int Engine::mark_move_done() {
  if (!ev_done_) PTB_CUDA_OK(cudaEventCreate(&ev_done_));
  PTB_CUDA_OK(cudaEventRecord(ev_done_, compute_));
  return 0;
}

// Direct path: every array is copied from the caller's memory as it is.
int Engine::move_direct(const double *origin, const double *dest, int8_t *flying, const double *weights,
                        int nchunks) {
  mirror_valid_ = false;  // the staging slots do not see this move
  cudaEvent_t ev_prev_done = chunk_events_[nchunks], ev_fly = chunk_events_[nchunks + 1];
  PTB_CUDA_OK(cudaStreamSynchronize(copy_));  // staged copies of an earlier move
  staged_chunks_ = 0;
  PTB_CUDA_OK(cudaEventRecord(ev_prev_done, compute_));
  PTB_CUDA_OK(cudaStreamWaitEvent(copy_, ev_prev_done, 0));
  if (!ev_copy0_) {
    PTB_CUDA_OK(cudaEventCreate(&ev_copy0_));
    PTB_CUDA_OK(cudaEventCreate(&ev_copy1_));
  }
  PTB_CUDA_OK(cudaEventRecord(ev_copy0_, copy_));
  PTB_CUDA_OK(cudaMemcpyAsync(d_flying_, flying, size_t(n_), cudaMemcpyHostToDevice, copy_));
  PTB_CUDA_OK(cudaEventRecord(ev_fly, copy_));
  for (int k = 0; k < nchunks; ++k) {
    const int32_t b = int32_t(int64_t(k) * chunk_), e = int32_t(std::min<int64_t>(n_, int64_t(b) + chunk_));
    const size_t cnt = size_t(e - b);
    PTB_CUDA_OK(cudaMemcpyAsync(d_origin_ + 3 * size_t(b), origin + 3 * size_t(b), 3 * cnt * sizeof(double), cudaMemcpyHostToDevice, copy_));
    PTB_CUDA_OK(cudaMemcpyAsync(d_dest_ + 3 * size_t(b), dest + 3 * size_t(b), 3 * cnt * sizeof(double), cudaMemcpyHostToDevice, copy_));
    PTB_CUDA_OK(cudaMemcpyAsync(d_weights_ + b, weights + b, cnt * sizeof(double), cudaMemcpyHostToDevice, copy_));
    PTB_CUDA_OK(cudaEventRecord(chunk_events_[k], copy_));
    PTB_CUDA_OK(cudaStreamWaitEvent(compute_, chunk_events_[k], 0));
    if (launch_range(d_origin_, d_dest_, d_flying_, d_weights_, b, e, compute_, true)) return 1;
  }
  PTB_CUDA_OK(cudaEventRecord(ev_copy1_, copy_));
  if (mark_move_done()) return 1;
  h2d_bytes_ += 57.0 * double(n_);
  stage_sent_bytes_ = 57.0 * double(n_);
  // reset the caller's flags once they are on the device (PumiTallyImpl.cpp:169-172)
  PTB_CUDA_OK(cudaEventSynchronize(ev_fly));
  if (n_) std::memset(flying, 0, size_t(n_));
  // caller may reuse its buffers on return (reference: blocking deep_copy)
  PTB_CUDA_OK(cudaStreamSynchronize(copy_));
  initial_weight_pending_ = false;
  ++moves_;
  return 0;
}

int Engine::move_to_next_location_device(const double *d_origin, const double *d_dest,
                                         const int8_t *d_flying, const double *d_weights,
                                         int32_t size, cudaStream_t stream) {
  if (int64_t(size) != 3 * int64_t(n_) || !initialized_) {
    fprintf(stderr, "[pumitally] ERROR: MoveToNextLocation(device): bad size or not initialised\n");
    return 1;
  }
  PTB_CUDA_OK(cudaSetDevice(device_));
  begin_move();
  // (the staging arrays are not touched: "pinned dest slots == device dest array" keeps holding, and the
  // next host move's origins are compared against them and patched exactly as after a host move)
  if (launch_range(d_origin, d_dest, d_flying, d_weights, 0, n_, stream, true)) return 1;
  initial_weight_pending_ = false;
  ++moves_;
  return 0;
}

// Score filter (SURVEY section 8 f4; OpenMC: an energy / material / ... filter on the tally).  nbins flux
// arrays of E doubles, bin-major, plus one unreported array for the particles no bin matches.
int Engine::set_score_bins(int32_t nbins) {
  if (nbins < 1 || nbins > 4096) return 1;
  if (nccl_comm_) {
    fprintf(stderr, "[pumitally] ERROR: set_score_bins after comm_init (the exchange buffers are sized by then)\n");
    return 1;
  }
  if (synchronize()) return 1;
  const size_t E = size_t(mesh_.ntets), len = size_t(nbins > 1 ? nbins + 1 : 1) * E + kFluxPad;
  double *nf = nullptr;
  PTB_CUDA_OK(cudaMalloc(reinterpret_cast<void **>(&nf), len * sizeof(double)));
  cudaFree(d_flux_);
  d_flux_ = nf;
  flux_alloc_ = len;
  nbins_ = nbins;
  release_batch_buffers();  // sized for the old number of bins
  if (nbins > 1 && !d_mask_) {
    PTB_CUDA_OK(cudaMalloc(reinterpret_cast<void **>(&d_mask_), std::max<size_t>(size_t(n_), 16)));
    PTB_CUDA_OK(cudaMalloc(reinterpret_cast<void **>(&d_bins_), std::max<size_t>(size_t(n_), 4) * sizeof(int32_t)));
  }
  return reset_tally();  // a new set of arrays starts from zero
}

// MoveToNextLocation with a score bin per particle for this move (host pointers).  bins == nullptr or one
// bin: the plain move.  The bins travel in one copy ahead of the particle data; everything else is the
// ordinary host path.
int Engine::move_to_next_location_binned(const double *origin, const double *dest, int8_t *flying, const double *weights,
                                         const int32_t *bins, int32_t size) {
  if (!bins || nbins_ == 1) return move_to_next_location(origin, dest, flying, weights, size);
  if (int64_t(size) != 3 * int64_t(n_) || !initialized_) return move_to_next_location(origin, dest, flying, weights, size);  // prints the error
  PTB_CUDA_OK(cudaSetDevice(device_));
  if (!ev_bins_) {
    PTB_CUDA_OK(cudaEventCreateWithFlags(&ev_bins_, cudaEventDisableTiming));
    PTB_CUDA_OK(cudaEventCreateWithFlags(&ev_bins_free_, cudaEventDisableTiming));
  }
  // d_bins_ is read by the mask kernels of the previous move until they are done
  PTB_CUDA_OK(cudaEventRecord(ev_bins_free_, compute_));
  PTB_CUDA_OK(cudaStreamWaitEvent(copy_, ev_bins_free_, 0));
  // through a pinned copy made by the worker pool (a pageable cudaMemcpyAsync of 40 MB blocks this thread for
  // milliseconds before the staging of the particle data can even start); the previous move's DMA out of it
  // was waited for before that move returned
  const int32_t *src = bins;
  if (!host_is_pinned(bins)) {
    if (!h_bins_ && cudaHostAlloc(reinterpret_cast<void **>(&h_bins_), std::max<size_t>(size_t(n_), 1) * sizeof(int32_t), cudaHostAllocDefault) != cudaSuccess) {
      cudaGetLastError();
      h_bins_ = nullptr;
    }
    if (h_bins_) {
      int32_t *dst = h_bins_;
      const size_t n = size_t(n_);
      if (stager_) {  // (the pool exists from the first staged move on)
        HostPool &pool = stager_->pool();
        const int T = pool.size();
        pool.run([&](int t) {
          const size_t lo = n * size_t(t) / size_t(T), hi = n * size_t(t + 1) / size_t(T);
          std::memcpy(dst + lo, bins + lo, (hi - lo) * sizeof(int32_t));
        });
      } else {
        std::memcpy(dst, bins, n * sizeof(int32_t));
      }
      src = h_bins_;
    }
  }
  PTB_CUDA_OK(cudaMemcpyAsync(d_bins_, src, size_t(n_) * sizeof(int32_t), cudaMemcpyHostToDevice, copy_));
  PTB_CUDA_OK(cudaEventRecord(ev_bins_, copy_));
  h2d_bytes_ += 4.0 * double(n_);
  cur_bins_ = d_bins_;
  // every pipeline stage is walked nbins + 1 times, seven small launches each, all enqueued by this thread between
  // two stage passes: unless the caller chose the stage size, binned moves use stages of 2 Mi particles
  const int32_t chunk = chunk_;
  if (!chunk_user_set_) chunk_ = std::max(chunk_, int32_t(1) << 21);
  const int rc = move_to_next_location(origin, dest, flying, weights, size);
  chunk_ = chunk;
  cur_bins_ = nullptr;
  PTB_CUDA_OK(cudaEventSynchronize(ev_bins_));  // the caller gets `bins` back with the other arrays
  return rc;
}

int Engine::move_to_next_location_device_binned(const double *d_origin, const double *d_dest, const int8_t *d_flying,
                                                const double *d_weights, const int32_t *d_bins, int32_t size,
                                                cudaStream_t stream) {
  cur_bins_ = (d_bins && nbins_ > 1) ? d_bins : nullptr;
  const int rc = move_to_next_location_device(d_origin, d_dest, d_flying, d_weights, size, stream);
  cur_bins_ = nullptr;
  return rc;
}

int Engine::synchronize() {
  PTB_CUDA_OK(cudaSetDevice(device_));
  PTB_CUDA_OK(cudaDeviceSynchronize());
  return 0;
}

int Engine::ensure_element_maps() {
  if (d_orig_of_internal_) return 0;
  const size_t E = std::max<size_t>(size_t(mesh_.ntets), 1);
  PTB_CUDA_OK(cudaMalloc(reinterpret_cast<void **>(&d_orig_of_internal_), E * sizeof(int32_t)));
  PTB_CUDA_OK(cudaMalloc(reinterpret_cast<void **>(&d_internal_of_orig_), E * sizeof(int32_t)));
  PTB_CUDA_OK(cudaMemcpy(d_orig_of_internal_, mesh_.orig_of_internal.data(), size_t(mesh_.ntets) * sizeof(int32_t), cudaMemcpyHostToDevice));
  PTB_CUDA_OK(cudaMemcpy(d_internal_of_orig_, mesh_.internal_of_orig.data(), size_t(mesh_.ntets) * sizeof(int32_t), cudaMemcpyHostToDevice));
  return 0;
}

// Places particles [first, first + count) at given positions in given elements (caller's numbering)
// without walking there: for drivers that hand particles between engines (spatial partition).  The
// elements are trusted to contain the positions.
int Engine::set_state_device(const double *d_xyz, const int32_t *d_elem, int32_t first, int32_t count, cudaStream_t stream) {
  if (first < 0 || count < 0 || int64_t(first) + count > n_) return 1;
  PTB_CUDA_OK(cudaSetDevice(device_));
  if (ensure_element_maps()) return 1;
  PTB_CUDA_OK(launch_set_state(d_state_, d_xyz, d_elem, d_internal_of_orig_, first, first + count, stream));
  initialized_ = true;
  mirror_valid_ = false;
  return 0;
}

int Engine::get_state_device(double *d_xyz, int32_t *d_elem, int32_t first, int32_t count, cudaStream_t stream) {
  if (first < 0 || count < 0 || int64_t(first) + count > n_) return 1;
  PTB_CUDA_OK(cudaSetDevice(device_));
  if (ensure_element_maps()) return 1;
  PTB_CUDA_OK(launch_get_state(d_state_, d_xyz, d_elem, d_orig_of_internal_, first, first + count, stream));
  return 0;
}

// (all score bins, bin-major: nbins * E values)
int Engine::get_flux_device(double *d_out, cudaStream_t stream) {
  PTB_CUDA_OK(cudaSetDevice(device_));
  if (ensure_element_maps() || gather_shares()) return 1;
  const size_t E = size_t(mesh_.ntets);
  for (int32_t b = 0; b < nbins_; ++b)
    PTB_CUDA_OK(launch_flux_to_caller_order(flux_view() + size_t(b) * E, d_orig_of_internal_, d_out + size_t(b) * E, mesh_.ntets, stream));
  return 0;
}

// n == E: the first (or only) score bin; n == nbins * E: every bin, bin-major
int Engine::get_flux(double *out, int64_t n) {
  const int64_t E = mesh_.ntets;
  if (n != E && n != int64_t(nbins_) * E) return 1;
  if (synchronize() || gather_shares()) return 1;
  std::vector<double> tmp(static_cast<size_t>(n));
  PTB_CUDA_OK(cudaMemcpy(tmp.data(), flux_view(), size_t(n) * sizeof(double), cudaMemcpyDeviceToHost));
  for (int64_t b = 0; b * E < n; ++b)
    for (int64_t i = 0; i < E; ++i) out[b * E + mesh_.orig_of_internal[i]] = tmp[b * E + i];  // caller's numbering
  return 0;
}

// NormalizeFlux (PumiTallyImpl.cpp:382-409); n as for get_flux (the volumes are always E values)
int Engine::get_normalized_flux(double *out_flux, double *out_volume, int64_t n) {
  const int64_t E = mesh_.ntets;
  if (n != E && n != int64_t(nbins_) * E) return 1;
  if (synchronize() || gather_shares()) return 1;
  if (out_flux) {
    const double per_source = source_normalization();
    if (!(per_source > 0.0)) {
      fprintf(stderr, "[pumitally] ERROR: source normalisation divisor is %g (no source weight seen yet?)\n", per_source);
      return 1;
    }
    std::vector<double> tmp(static_cast<size_t>(E));
    for (int64_t b = 0; b * E < n; ++b) {
      PTB_CUDA_OK(launch_normalize(flux_view() + size_t(b * E), d_volume_, d_scratch_, E, per_source, compute_));
      PTB_CUDA_OK(cudaStreamSynchronize(compute_));
      PTB_CUDA_OK(cudaMemcpy(tmp.data(), d_scratch_, size_t(E) * sizeof(double), cudaMemcpyDeviceToHost));
      for (int64_t i = 0; i < E; ++i) out_flux[b * E + mesh_.orig_of_internal[i]] = tmp[i];
    }
  }
  if (out_volume)
    for (int64_t i = 0; i < E; ++i) out_volume[mesh_.orig_of_internal[i]] = mesh_.volume[i];
  return 0;
}

int Engine::get_element_ids(int32_t *out, int64_t n) {
  if (n != n_) return 1;
  if (synchronize()) return 1;
  std::vector<ParticleState> tmp(static_cast<size_t>(n_));
  PTB_CUDA_OK(cudaMemcpy(tmp.data(), d_state_, size_t(n_) * sizeof(ParticleState), cudaMemcpyDeviceToHost));
  for (int64_t i = 0; i < n_; ++i) out[i] = mesh_.orig_of_internal[tmp[i].elem];  // caller's numbering
  return 0;
}

int Engine::get_positions(double *out, int64_t n3) {
  if (n3 != 3 * int64_t(n_)) return 1;
  if (synchronize()) return 1;
  std::vector<ParticleState> tmp(static_cast<size_t>(n_));
  PTB_CUDA_OK(cudaMemcpy(tmp.data(), d_state_, size_t(n_) * sizeof(ParticleState), cudaMemcpyDeviceToHost));
  for (int64_t i = 0; i < n_; ++i) {
    out[3 * i] = tmp[i].x;
    out[3 * i + 1] = tmp[i].y;
    out[3 * i + 2] = tmp[i].z;
  }
  return 0;
}

int Engine::set_source_normalization(int mode, double value) {
  if (mode < 0 || mode > 3 || (mode == 2 && !(value > 0.0))) return 1;
  norm_mode_ = mode;
  norm_value_ = value;
  return 0;
}

double Engine::source_normalization() {
  switch (norm_mode_) {
    case 1: return double(std::max(n_, 1));
    case 2: return norm_value_;
    case 3: {
      double w = 0.0;
      cudaDeviceSynchronize();
      if (cudaMemcpy(&w, d_initial_weight_, sizeof(double), cudaMemcpyDeviceToHost) != cudaSuccess) return 0.0;
      return w;
    }
    default: return 1.0;
  }
}

int Engine::reset_tally() {
  if (synchronize()) return 1;
  collect_timers(true);
  PTB_CUDA_OK(cudaMemset(d_initial_weight_, 0, sizeof(double)));
  initial_weight_pending_ = true;
  PTB_CUDA_OK(cudaMemset(d_flux_, 0, flux_alloc_ * sizeof(double)));
  PTB_CUDA_OK(cudaMemset(d_stats_, 0, sizeof(DeviceStats)));
  flux_global_valid_ = flux_owned_only_ = false;
  kernel_ms_ = 0.0;
  h2d_bytes_ = 0.0;
  moves_ = 0;
  batches_ = 0;  // the next end_batch starts the sums over (no need to clear them)
  return 0;
}

int Engine::get_stats(EngineStats *out) {
  if (synchronize()) return 1;
  collect_timers(true);
  DeviceStats s;
  PTB_CUDA_OK(cudaMemcpy(&s, d_stats_, sizeof(s), cudaMemcpyDeviceToHost));
  out->segments = s.segments;
  out->tracks = s.tracks;
  out->relocations = s.relocations;
  out->lost = s.lost;
  out->moves = moves_;
  out->kernel_ms = kernel_ms_;
  out->h2d_bytes = h2d_bytes_;
  out->plane_fallbacks = s.fallbacks;
  if (s.lost)  // reference wording, PumiTallyImpl.cpp:455-458
    printf("ERROR: Not all particles are found. May need more loops in search\n");
  return 0;
}

// The tet table of config c2 (128 MB) still half-fits the L2, and streaming the particles in
// storage order through the TMA stages is fastest.  Once the table is several times the L2
// (config c5: 1.26 GB) nearly every record fetch is a random 32-byte DRAM access; processing the
// particles in spatial order (binning pass + gather staging) then pays for itself twice over
// (profiles/r01/README.md, section q).
int Engine::choose_variant() const {
  int l2 = 0;
  cudaDeviceGetAttribute(&l2, cudaDevAttrL2CacheSize, device_);
  const double table = double(mesh_.ntets) * sizeof(TetRecord);
  return (l2 > 0 && table > 2.0 * double(l2)) ? kVariantPersistGatherL1 : kVariantPersistRefill8;
}

int64_t Engine::get_option(const std::string &name) const {
  if (name == "variant")  // the kernel the next move will use outside the auto-tuner's exploration moves
    return (auto_variant_ && autotune_ && variant_ == kVariantPersistRefill8) ? tuned_variant_ : variant_;
  if (name == "launches") return int64_t(launches_);
  if (name == "autotune") return autotune_ ? 1 : 0;
  if (name == "block") return block_;
  if (name == "chunk") return chunk_;
  if (name == "seed_grid") return seed_grid_mode_;
  if (name == "seed_grid_active") return use_seed_grid_ ? 1 : 0;
  if (name == "hull_convex") return mesh_.hull_convex ? 1 : 0;
  if (name == "max_iters") return max_iters_;
  if (name == "l2_fetch") {
    size_t g = 0;
    return cudaDeviceGetLimit(&g, cudaLimitMaxL2FetchGranularity) == cudaSuccess ? int64_t(g) : -1;
  }
  if (name == "allreduce_us") return int64_t(allreduce_ms_ * 1e3);  // device time of the last batch-end exchange
  if (name == "score_bins") return nbins_;
  if (name == "batches") return int64_t(batches_);  // batches closed by end_batch since the last reset
  if (name == "exchange_choice") return exchange_choice_;  // what exchange_tally() does: 0 all-reduce, 1 reduce-scatter
  if (name == "exchange_allreduce_us") return int64_t(exchange_ms_[0] * 1e3);  // comm_init's measurement of the two
  if (name == "exchange_reduce_scatter_us") return int64_t(exchange_ms_[1] * 1e3);
  if (name == "host_path") return host_path_;
  if (name == "host_path_last") return span_tag_ == 1 ? 0 : 1;  // path of the last host move: 1 staged, 0 direct
  if (name == "host_threads") return stager_ ? stager_->threads() : host_threads_;
  if (name == "stage_host_us") return int64_t(stage_host_s_ * 1e6);   // last staged move: host time from entry to return
  if (name == "stage_sent_bytes") return int64_t(stage_sent_bytes_);  // last staged move: bytes put on the wire
  if (name == "staged") return stage_ready_ ? 1 : 0;
  if (name == "stage_copy_us") {  // last staged move: device time from "copy stream free" to the last upload's end
    float ms = 0.f;
    if (!ev_copy0_ || cudaEventSynchronize(ev_copy1_) != cudaSuccess || cudaEventElapsedTime(&ms, ev_copy0_, ev_copy1_) != cudaSuccess) {
      cudaGetLastError();
      return -1;
    }
    return int64_t(ms * 1e3);
  }
  if (name == "host_node") return pool_node_;  // NUMA node the staging workers run on (-1: not pinned to one)
  return -1;
}

int Engine::set_option(const std::string &name, int64_t v) {
  if (name == "variant") {
    if (v == -1) {  // automatic
      variant_ = choose_variant();
      auto_variant_ = true;
      return 0;
    }
    if (v < 0 || v >= kNumVariants || !walk_variant_available(int(v))) return 1;
    if (v >= kVariantEdge && v <= kVariantEdgeOcc6) {
      if (synchronize()) return 1;
      try {
        if (!upload_compact()) return 1;
      } catch (const std::exception &ex) {
        fprintf(stderr, "%s\n", ex.what());
        return 1;
      }
    }
    variant_ = int(v);
    auto_variant_ = false;
  } else if (name == "autotune") {
    autotune_ = v != 0;
  } else if (name == "block") {
    if (v != 64 && v != 128 && v != 256) return 1;
    block_ = int(v);
  } else if (name == "chunk") {
    if (v < 1024) return 1;
    chunk_ = int32_t(std::min<int64_t>(v, INT_MAX)) & ~1023;  // keeps every range 16-byte aligned
    chunk_user_set_ = true;
  } else if (name == "exchange_choice") {
    exchange_choice_ = v ? 1 : 0;  // the caller must set the same value on every rank
  } else if (name == "seed_grid") {
    if (v < 0 || v > 2) return 1;
    seed_grid_mode_ = int(v);
    use_seed_grid_ = v == 2 || (v == 1 && mesh_.hull_convex);
  } else if (name == "register_host") {
    register_host_ = v != 0;
  } else if (name == "max_iters") {  // crossing limit per walk (the tracer's loop limit); 0 = number of tets + 16
    if (v < 0 || v > INT_MAX) return 1;
    max_iters_ = int32_t(v);
  } else if (name == "l2_fetch") {  // bytes an L2 miss fetches from DRAM: 32, 64 or 128 (device-wide limit)
    if (v != 32 && v != 64 && v != 128) return 1;
    if (cudaDeviceSetLimit(cudaLimitMaxL2FetchGranularity, size_t(v)) != cudaSuccess) { cudaGetLastError(); return 1; }
  } else if (name == "host_path") {  // 2 = automatic (default), 1 = staged through the pinned slots, 0 = direct copies
    if (v < 0 || v > 2) return 1;
    host_path_ = int(v);
    if (host_path_ == 0) mirror_valid_ = false;
  } else if (name == "host_threads") {  // workers of the staging pool; before the first host-pointer call
    if (v < 1 || v > 256 || stager_) return 1;
    host_threads_ = int(v);
  } else if (name == "morton") {
    morton_ = v != 0;
  } else if (name == "claim_run") {
    if (v != 1 && v != 2 && v != 4) return 1;
    claim_run_ = int(v);
  } else {
    return 1;
  }
  return 0;
}

int64_t Engine::debug_order(int32_t *out, int64_t n) {
  if (!last_work_count_ || synchronize()) return -1;
  unsigned int cnt = 0;
  if (cudaMemcpy(&cnt, last_work_count_, sizeof(cnt), cudaMemcpyDeviceToHost) != cudaSuccess) return -1;
  const int64_t m = std::min<int64_t>(n, cnt);
  if (m > 0 && cudaMemcpy(out, d_order_, size_t(m) * sizeof(int32_t), cudaMemcpyDeviceToHost) != cudaSuccess) return -1;
  return cnt;
}

// FinalizeTallies (PumiTallyImpl.cpp:411-416)
int Engine::write_tally_results() {
  const size_t E = size_t(mesh_.ntets);
  std::vector<double> nf(E * size_t(nbins_)), vol(E), sd;
  if (batches_ > 0) {
    // after end_batch: the mean over the ended batches (moves since the last one are not part of the result)
    // and, from two batches on, its standard deviation
    if (batches_ >= 2) sd.resize(nf.size());
    if (get_tally_statistics(nf.data(), sd.empty() ? nullptr : sd.data(), int64_t(nf.size()))) return 1;
    for (size_t i = 0; i < E; ++i) vol[mesh_.orig_of_internal[i]] = mesh_.volume[i];
  } else if (get_normalized_flux(nf.data(), vol.data(), int64_t(nf.size()))) {  // caller's element order
    return 1;
  }
  // filtered tally: "flux" is the sum over the bins (what the unfiltered tally would hold), and every
  // bin is written as "flux_bin<k>" next to it (the sum gets no standard deviation: that would need the
  // covariances between the bins)
  std::vector<std::pair<std::string, const double *>> extra;
  std::vector<double> per_bin;
  if (nbins_ > 1) {
    per_bin.assign(nf.begin(), nf.end());
    for (int32_t b = 0; b < nbins_; ++b) {
      extra.emplace_back("flux_bin" + std::to_string(b), per_bin.data() + size_t(b) * E);
      if (!sd.empty()) extra.emplace_back("flux_bin" + std::to_string(b) + "_std_dev", sd.data() + size_t(b) * E);
    }
    for (int32_t b = 1; b < nbins_; ++b)
      for (size_t i = 0; i < E; ++i) nf[i] += nf[size_t(b) * E + i];
    nf.resize(E);
  } else if (!sd.empty()) {
    extra.emplace_back("flux_std_dev", sd.data());
  }
  std::string err;
  if (!write_vtk_dataset(output_name_, mesh_, nf, vol, rank_, nranks_, &err, extra)) {
    fprintf(stderr, "[pumitally] ERROR: %s\n", err.c_str());
    return 1;
  }
  return 0;
}

// ------------------------------------------------------------------ batch statistics

size_t Engine::stats_count() const {
  const size_t off = stats_offset(), len = flux_len();
  return off >= len ? 0 : std::min(stats_len(), len - off);
}

// Allocated at the first end_batch, so that engines that never end a batch keep their memory footprint.
int Engine::ensure_batch_buffers() {
  if (d_s1_) return 0;
  const size_t len = std::max<size_t>(stats_len(), 1);
  const size_t small = 3 * size_t(kBatchTriggerBlocks) + 3 + 3 * size_t(std::max(nranks_, 1)) + 2;
  if (cudaMalloc(reinterpret_cast<void **>(&d_s1_), len * sizeof(double)) != cudaSuccess ||
      cudaMalloc(reinterpret_cast<void **>(&d_s2_), len * sizeof(double)) != cudaSuccess ||
      cudaMalloc(reinterpret_cast<void **>(&d_batch_small_), small * sizeof(double)) != cudaSuccess) {
    cudaGetLastError();
    fprintf(stderr, "[pumitally] ERROR: no device memory for the batch statistics (%zu MB)\n", (2 * len * sizeof(double)) >> 20);
    release_batch_buffers();
    return 1;
  }
  batches_ = 0;
  return 0;
}

void Engine::release_batch_buffers() {
  cudaFree(d_s1_);
  cudaFree(d_s2_);
  cudaFree(d_batch_small_);
  d_s1_ = d_s2_ = d_batch_small_ = nullptr;
  batches_ = 0;
}

// The batch's source divisor: 1 (mode 0), the number of particles (1), the caller's value (2: the global
// source weight of one batch), the weight of the batch's first tracks (3).  Particles and weights are summed
// over the ranks (collective), unlike get_normalized_flux's per-rank divisor.
int Engine::batch_divisor(double *out) {
  double v = 1.0;
  if (norm_mode_ == 1) v = double(n_);
  else if (norm_mode_ == 2) v = norm_value_;
  else if (norm_mode_ == 3) PTB_CUDA_OK(cudaMemcpy(&v, d_initial_weight_, sizeof(double), cudaMemcpyDeviceToHost));
  if (nccl_comm_ && (norm_mode_ == 1 || norm_mode_ == 3)) {
    double *d = d_batch_small_ + 3 * size_t(kBatchTriggerBlocks) + 3 + 3 * size_t(nranks_);
    PTB_CUDA_OK(cudaMemcpyAsync(d, &v, sizeof(double), cudaMemcpyHostToDevice, compute_));
    if (nccl_allreduce_sum_f64(nccl_comm_, d, d + 1, 1, compute_)) return 1;
    PTB_CUDA_OK(cudaMemcpyAsync(&v, d + 1, sizeof(double), cudaMemcpyDeviceToHost, compute_));
    PTB_CUDA_OK(cudaStreamSynchronize(compute_));
  }
  *out = v;
  return 0;
}

// Ordering: the device synchronisation at the start puts every kernel of earlier moves, on whichever stream
// they were enqueued, before the accumulate pass, and the pass has finished when the call returns, so every
// later move comes after it.
int Engine::end_batch() {
  PTB_CUDA_OK(cudaSetDevice(device_));
  if (synchronize() || ensure_batch_buffers()) return 1;
  double div = 0.0;
  if (batch_divisor(&div)) return 1;
  if (!(std::isfinite(div) && div > 0.0)) {
    fprintf(stderr, "[pumitally] ERROR: end_batch: the batch's source divisor (normalisation mode %d) is %g%s; "
                    "nothing was accumulated\n", norm_mode_, div,
            norm_mode_ == 3 ? " (no flying particle with a weight in the batch's first move)" : "");
    return 1;
  }
  const double *x = d_flux_;
  double *zero = d_flux_;  // one GPU: the pass clears the tally it reads
  if (nccl_comm_) {
    if (exchange_tally()) return 1;
    x = d_flux_global_ + stats_offset();  // this rank's share of the sum over ranks
    zero = nullptr;
    PTB_CUDA_OK(cudaMemsetAsync(d_flux_, 0, flux_alloc_ * sizeof(double), compute_));
  } else if (flux_alloc_ > flux_len()) {  // the unreported bin and the pad
    PTB_CUDA_OK(cudaMemsetAsync(d_flux_ + flux_len(), 0, (flux_alloc_ - flux_len()) * sizeof(double), compute_));
  }
  PTB_CUDA_OK(launch_batch_accumulate(x, div, zero, d_s1_, d_s2_, int64_t(stats_count()), batches_ == 0, compute_));
  PTB_CUDA_OK(cudaMemsetAsync(d_initial_weight_, 0, sizeof(double), compute_));
  PTB_CUDA_OK(cudaStreamSynchronize(compute_));
  initial_weight_pending_ = true;
  flux_global_valid_ = flux_owned_only_ = false;
  ++batches_;
  return 0;
}

int Engine::get_tally_statistics(double *out_mean, double *out_std_dev, int64_t n) {
  const int64_t E = mesh_.ntets;
  if (n != E && n != int64_t(nbins_) * E) return 1;
  if (batches_ == 0) {
    fprintf(stderr, "[pumitally] ERROR: tally statistics before the first end_batch\n");
    return 1;
  }
  if (synchronize()) return 1;
  // the finish pass writes this rank's share of both arrays, the all-gather (collective) the others
  const size_t full = nccl_comm_ ? share_ * size_t(nranks_) : flux_len(), off = stats_offset();
  double *d_out = nullptr;
  PTB_CUDA_OK(cudaMalloc(reinterpret_cast<void **>(&d_out), 2 * std::max<size_t>(full, 1) * sizeof(double)));
  std::unique_ptr<double, cudaError_t (*)(void *)> keep(d_out, cudaFree);
  double *d_mean = d_out, *d_std = d_out + full;
  PTB_CUDA_OK(launch_batch_finish(d_s1_, d_s2_, int64_t(stats_count()), int64_t(off), E, d_volume_, double(batches_),
                                  d_mean + off, d_std + off, compute_));
  if (nccl_comm_ && (nccl_all_gather_f64(nccl_comm_, d_mean + off, d_mean, share_, compute_) ||
                     nccl_all_gather_f64(nccl_comm_, d_std + off, d_std, share_, compute_)))
    return 1;
  PTB_CUDA_OK(cudaStreamSynchronize(compute_));
  std::vector<double> tmp(static_cast<size_t>(n));
  const std::pair<double *, const double *> outs[2] = {{out_mean, d_mean}, {out_std_dev, d_std}};
  for (const auto &o : outs) {
    if (!o.first) continue;
    PTB_CUDA_OK(cudaMemcpy(tmp.data(), o.second, size_t(n) * sizeof(double), cudaMemcpyDeviceToHost));
    for (int64_t b = 0; b * E < n; ++b)
      for (int64_t i = 0; i < E; ++i) o.first[b * E + mesh_.orig_of_internal[i]] = tmp[b * E + i];  // caller's numbering
  }
  return 0;
}

// Tally trigger: each rank reduces its share to one (max, index, count) record, the records are gathered
// and combined the same way on every rank.
int Engine::max_relative_error(double threshold, double *max_rel, int64_t *index, int64_t *count_above) {
  if (batches_ < 2) {
    fprintf(stderr, "[pumitally] ERROR: the relative error needs at least two ended batches (have %llu)\n",
            (unsigned long long)batches_);
    return 1;
  }
  if (synchronize() || ensure_element_maps()) return 1;
  double *rec = d_batch_small_ + 3 * size_t(kBatchTriggerBlocks), *all = rec + 3;
  PTB_CUDA_OK(launch_batch_trigger(d_s1_, d_s2_, int64_t(stats_count()), int64_t(stats_offset()), mesh_.ntets,
                                   d_volume_, d_orig_of_internal_, double(batches_), threshold, d_batch_small_, rec,
                                   compute_));
  const int nrec = nccl_comm_ ? nranks_ : 1;
  if (nccl_comm_ && nccl_all_gather_f64(nccl_comm_, rec, all, 3, compute_)) return 1;
  std::vector<double> h(3 * size_t(nrec));
  PTB_CUDA_OK(cudaMemcpyAsync(h.data(), nccl_comm_ ? all : rec, h.size() * sizeof(double), cudaMemcpyDeviceToHost, compute_));
  PTB_CUDA_OK(cudaStreamSynchronize(compute_));
  double best = -1.0, cnt = 0.0;
  int64_t best_idx = -1;
  for (int r = 0; r < nrec; ++r) {
    const double rel = h[3 * size_t(r)];
    const int64_t idx = int64_t(h[3 * size_t(r) + 1]);
    cnt += h[3 * size_t(r) + 2];
    if (rel >= 0.0 && (rel > best || (rel == best && idx < best_idx))) {
      best = rel;
      best_idx = idx;
    }
  }
  if (max_rel) *max_rel = best < 0.0 ? 0.0 : best;
  if (index) *index = best_idx;
  if (count_above) *count_above = int64_t(cnt);
  return 0;
}

// ------------------------------------------------------------------ multi-GPU

int Engine::comm_init(int rank, int nranks, const uint8_t id[128]) {
  PTB_CUDA_OK(cudaSetDevice(device_));
  if (nccl_comm_) return 1;
  if (nccl_comm_init_rank(&nccl_comm_, nranks, id, rank)) return 1;
  rank_ = rank;
  nranks_ = nranks;
  release_batch_buffers();  // from here on every rank keeps the statistics of its share only
  // NCCL sets up its NVLink connections lazily inside the first collective: pay that here,
  // on the scratch array, not in the first batch-end exchange
  if (nranks < 1 || size_t(nranks) > kFluxPad) return 1;
  share_ = (flux_len() + size_t(nranks) - 1) / size_t(nranks);
  PTB_CUDA_OK(cudaMalloc(reinterpret_cast<void **>(&d_flux_global_), std::max<size_t>(share_ * size_t(nranks), 1) * sizeof(double)));
  PTB_CUDA_OK(cudaEventCreate(&ev_ar0_));
  PTB_CUDA_OK(cudaEventCreate(&ev_ar1_));
  PTB_CUDA_OK(cudaMemsetAsync(d_scratch_, 0, size_t(mesh_.ntets) * sizeof(double), compute_));
  if (nccl_allreduce_sum_f64(nccl_comm_, d_scratch_, d_flux_global_, size_t(mesh_.ntets), compute_)) return 1;
  // ... and so does every other collective the first time it is used (measured: 0.86 s for the first
  // ncclReduceScatter on 8 GPUs): warm up the reduce-scatter / all-gather pair of reduce_tally_to_owners too.
  // d_flux_ is all zeros here or holds this rank's tally, which the exchange does not modify.
  if (nccl_reduce_scatter_sum_f64(nccl_comm_, d_flux_, d_flux_global_ + size_t(rank_) * share_, share_, compute_)) return 1;
  if (nccl_all_gather_f64(nccl_comm_, d_flux_global_ + size_t(rank_) * share_, d_flux_global_, share_, compute_)) return 1;
  PTB_CUDA_OK(cudaStreamSynchronize(compute_));
  // Which of the two batch-end exchanges is quicker depends on the array size and on what NCCL picks for it
  // (measured on 8 B200s: 8 MB of flux -- all-reduce 0.10 ms, reduce-scatter 4.3 ms; 79 MB -- 0.9 ms and 0.43 ms):
  // time both on this mesh and let exchange_tally() use the quicker one.  The times are summed over the ranks
  // so that every rank takes the same decision.
  double t[2] = {1e30, 1e30};
  for (int rep = 0; rep < 3; ++rep)
    for (int which = 0; which < 2; ++which) {
      PTB_CUDA_OK(cudaEventRecord(ev_ar0_, compute_));
      if (which == 0 ? nccl_allreduce_sum_f64(nccl_comm_, d_flux_, d_flux_global_, flux_len(), compute_)
                     : nccl_reduce_scatter_sum_f64(nccl_comm_, d_flux_, d_flux_global_ + size_t(rank_) * share_, share_, compute_))
        return 1;
      PTB_CUDA_OK(cudaEventRecord(ev_ar1_, compute_));
      PTB_CUDA_OK(cudaStreamSynchronize(compute_));
      float ms = 0.f;
      PTB_CUDA_OK(cudaEventElapsedTime(&ms, ev_ar0_, ev_ar1_));
      t[which] = std::min(t[which], double(ms));
    }
  double *d_t = d_scratch_;  // E >= 2 doubles of scratch: meshes have more than two elements
  if (mesh_.ntets < 4) { exchange_choice_ = 0; return 0; }
  PTB_CUDA_OK(cudaMemcpyAsync(d_t, t, sizeof(t), cudaMemcpyHostToDevice, compute_));
  if (nccl_allreduce_sum_f64(nccl_comm_, d_t, d_t + 2, 2, compute_)) return 1;
  PTB_CUDA_OK(cudaMemcpyAsync(t, d_t + 2, sizeof(t), cudaMemcpyDeviceToHost, compute_));
  PTB_CUDA_OK(cudaStreamSynchronize(compute_));
  exchange_ms_[0] = t[0] / nranks;
  exchange_ms_[1] = t[1] / nranks;
  exchange_choice_ = t[1] < t[0] ? 1 : 0;
  return 0;
}

// The batch-end exchange this mesh and this machine do quickest (chosen in comm_init)
int Engine::exchange_tally() { return exchange_choice_ == 1 ? reduce_tally_to_owners() : allreduce_tally(); }

// Batch-end exchange: sum the per-rank tallies.  Every rank holds a full-buffer
// picpart (all elements are ghosts of every other rank), so the ghost-layer
// array is the whole flux array.  Out of place: d_flux_ stays this rank's own running tally, the
// sum over ranks lands in d_flux_global_ -- the call may be repeated after every batch.
int Engine::allreduce_tally() {
  if (!nccl_comm_) return nranks_ == 1 ? 0 : 1;
  PTB_CUDA_OK(cudaSetDevice(device_));
  PTB_CUDA_OK(cudaDeviceSynchronize());
  PTB_CUDA_OK(cudaEventRecord(ev_ar0_, compute_));
  if (nccl_allreduce_sum_f64(nccl_comm_, d_flux_, d_flux_global_, flux_len(), compute_)) return 1;
  PTB_CUDA_OK(cudaEventRecord(ev_ar1_, compute_));
  PTB_CUDA_OK(cudaStreamSynchronize(compute_));
  float ms = 0.f;
  if (cudaEventElapsedTime(&ms, ev_ar0_, ev_ar1_) == cudaSuccess) allreduce_ms_ = ms;
  flux_global_valid_ = true;
  flux_owned_only_ = false;
  return 0;
}

int Engine::reduce_tally_to_owners() {
  if (!nccl_comm_) return nranks_ == 1 ? 0 : 1;
  PTB_CUDA_OK(cudaSetDevice(device_));
  PTB_CUDA_OK(cudaDeviceSynchronize());
  PTB_CUDA_OK(cudaEventRecord(ev_ar0_, compute_));
  if (nccl_reduce_scatter_sum_f64(nccl_comm_, d_flux_, d_flux_global_ + size_t(rank_) * share_, share_, compute_)) return 1;
  PTB_CUDA_OK(cudaEventRecord(ev_ar1_, compute_));
  PTB_CUDA_OK(cudaStreamSynchronize(compute_));
  float ms = 0.f;
  if (cudaEventElapsedTime(&ms, ev_ar0_, ev_ar1_) == cudaSuccess) allreduce_ms_ = ms;
  flux_global_valid_ = true;
  flux_owned_only_ = true;
  return 0;
}

// Collective: every rank contributes its share, every rank ends up with the whole (summed) array.
int Engine::gather_shares() {
  if (!flux_global_valid_ || !flux_owned_only_) return 0;
  PTB_CUDA_OK(cudaSetDevice(device_));
  if (nccl_all_gather_f64(nccl_comm_, d_flux_global_ + size_t(rank_) * share_, d_flux_global_, share_, compute_)) return 1;
  PTB_CUDA_OK(cudaStreamSynchronize(compute_));
  flux_owned_only_ = false;
  return 0;
}

}  // namespace ptb
