// extern "C" layer of libpumitally.so (declarations and reference citations in
// include/pumitally_c.h).  No exceptions cross this boundary.
#include "pumitally_c.h"

#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <exception>
#include <string>

#include "engine.hpp"

struct pumitally_engine {
  ptb::Engine *impl;
};

namespace {

int device_from_args(int *argc, char ***argv) {
  int dev = -1;
  if (const char *env = std::getenv("PUMITALLY_DEVICE")) dev = std::atoi(env);
  if (argc && argv && *argv)
    for (int i = 0; i < *argc; ++i) {
      const char *a = (*argv)[i];
      if (a && std::strncmp(a, "--pumitally-device=", 19) == 0) dev = std::atoi(a + 19);
    }
  return dev;
}

pumitally_engine *make_engine(ptb::HostMesh &&mesh, int32_t num_particles, int device) {
  try {
    auto *h = new pumitally_engine{nullptr};
    h->impl = new ptb::Engine(std::move(mesh), num_particles, device);
    return h;
  } catch (const std::exception &ex) {
    fprintf(stderr, "%s\n", ex.what());
    return nullptr;
  }
}

template <typename F>
int guarded(pumitally_engine *e, F &&f) {
  if (!e || !e->impl) {
    fprintf(stderr, "[pumitally] ERROR: null engine handle\n");
    return 1;
  }
  try {
    return f(*e->impl);
  } catch (const std::exception &ex) {
    fprintf(stderr, "[pumitally] ERROR: %s\n", ex.what());
    return 1;
  }
}

}  // namespace

extern "C" {

pumitally_engine *pumitally_create(const char *mesh_filename, int32_t num_particles, int *argc,
                                   char ***argv) {
  // reference prints the same banner (PumiTallyImpl.cpp:554-555)
  printf("Reading the Omega_h mesh %s to tally with tracklength estimator\n",
         mesh_filename ? mesh_filename : "");
  ptb::HostMesh mesh;
  std::string err;
  if (!mesh.load(mesh_filename ? mesh_filename : "", &err)) {
    fprintf(stderr, "[ERROR] %s\n", err.c_str());
    return nullptr;
  }
  printf("PumiPIC Loaded mesh %s with %lld elements\n", mesh_filename, (long long)mesh.ntets);
  return make_engine(std::move(mesh), num_particles, device_from_args(argc, argv));
}

pumitally_engine *pumitally_create_from_arrays(const double *coords, int64_t nverts,
                                               const int32_t *tet2vert, int64_t ntets,
                                               int32_t num_particles, int32_t device) {
  ptb::HostMesh mesh;
  std::string err;
  if (!mesh.from_arrays(coords, nverts, tet2vert, ntets, &err)) {
    fprintf(stderr, "[ERROR] %s\n", err.c_str());
    return nullptr;
  }
  if (device < 0) device = device_from_args(nullptr, nullptr);
  return make_engine(std::move(mesh), num_particles, device);
}

int pumitally_copy_initial_position(pumitally_engine *e, const double *xyz, int32_t size) {
  if (size > 0 && !xyz) {
    fprintf(stderr, "[pumitally] ERROR: CopyInitialPosition: null position array\n");
    return 1;
  }
  return guarded(e, [&](ptb::Engine &g) { return g.copy_initial_position(xyz, size); });
}

int pumitally_move_to_next_location(pumitally_engine *e, const double *origin, const double *dest,
                                    int8_t *flying, const double *weights, int32_t size) {
  if (size > 0 && (!origin || !dest || !flying || !weights)) {
    fprintf(stderr, "[pumitally] ERROR: MoveToNextLocation: null input array\n");
    return 1;
  }
  return guarded(e, [&](ptb::Engine &g) {
    return g.move_to_next_location(origin, dest, flying, weights, size);
  });
}

int pumitally_write_tally_results(pumitally_engine *e) {
  return guarded(e, [&](ptb::Engine &g) { return g.write_tally_results(); });
}

void pumitally_destroy(pumitally_engine *e) {
  if (!e) return;
  delete e->impl;
  delete e;
}

int64_t pumitally_num_elements(const pumitally_engine *e) {
  return (e && e->impl) ? e->impl->num_elements() : -1;
}
int32_t pumitally_num_particles(const pumitally_engine *e) {
  return (e && e->impl) ? e->impl->num_particles() : -1;
}
int pumitally_get_flux(pumitally_engine *e, double *out, int64_t n) {
  return guarded(e, [&](ptb::Engine &g) { return g.get_flux(out, n); });
}
int pumitally_get_normalized_flux(pumitally_engine *e, double *out_flux, double *out_volume,
                                  int64_t n) {
  return guarded(e, [&](ptb::Engine &g) { return g.get_normalized_flux(out_flux, out_volume, n); });
}
int pumitally_get_element_ids(pumitally_engine *e, int32_t *out, int64_t n) {
  return guarded(e, [&](ptb::Engine &g) { return g.get_element_ids(out, n); });
}
int pumitally_get_positions(pumitally_engine *e, double *out, int64_t n3) {
  return guarded(e, [&](ptb::Engine &g) { return g.get_positions(out, n3); });
}
int pumitally_get_adjacency(const pumitally_engine *e, int32_t *out, int64_t n4) {
  if (!e || !e->impl || n4 != 4 * e->impl->num_elements()) return 1;
  const std::vector<int32_t> adj = e->impl->mesh().adjacency_original();
  std::memcpy(out, adj.data(), size_t(n4) * sizeof(int32_t));
  return 0;
}
int pumitally_set_score_bins(pumitally_engine *e, int32_t nbins) {
  return guarded(e, [&](ptb::Engine &g) { return g.set_score_bins(nbins); });
}
int32_t pumitally_get_score_bins(const pumitally_engine *e) {
  return e ? int32_t(pumitally_get_option(e, "score_bins")) : 0;
}
int pumitally_move_to_next_location_binned(pumitally_engine *e, const double *origin, const double *dest,
                                           int8_t *flying, const double *weights, const int32_t *bins, int32_t size) {
  if (size > 0 && (!origin || !dest || !flying || !weights)) {
    fprintf(stderr, "[pumitally] ERROR: MoveToNextLocation: null input array\n");
    return 1;
  }
  return guarded(e, [&](ptb::Engine &g) { return g.move_to_next_location_binned(origin, dest, flying, weights, bins, size); });
}
int pumitally_move_to_next_location_device_binned(pumitally_engine *e, const double *d_origin, const double *d_dest,
                                                  const int8_t *d_flying, const double *d_weights, const int32_t *d_bins,
                                                  int32_t size, void *stream) {
  return guarded(e, [&](ptb::Engine &g) {
    return g.move_to_next_location_device_binned(d_origin, d_dest, d_flying, d_weights, d_bins, size,
                                                 static_cast<cudaStream_t>(stream));
  });
}

int pumitally_reset_tally(pumitally_engine *e) {
  return guarded(e, [&](ptb::Engine &g) { return g.reset_tally(); });
}

int pumitally_set_source_normalization(pumitally_engine *e, int32_t mode, double value) {
  return guarded(e, [&](ptb::Engine &g) { return g.set_source_normalization(mode, value); });
}
double pumitally_get_source_normalization(pumitally_engine *e) {
  return (e && e->impl) ? e->impl->source_normalization() : 0.0;
}

int pumitally_get_stats(pumitally_engine *e, pumitally_stats *out) {
  return guarded(e, [&](ptb::Engine &g) {
    ptb::EngineStats s;
    if (g.get_stats(&s)) return 1;
    out->segments = s.segments;
    out->tracks = s.tracks;
    out->relocations = s.relocations;
    out->lost = s.lost;
    out->moves = s.moves;
    out->kernel_ms = s.kernel_ms;
    out->h2d_bytes = s.h2d_bytes;
    out->plane_fallbacks = s.plane_fallbacks;
    return 0;
  });
}

int pumitally_set_output_name(pumitally_engine *e, const char *filename) {
  return guarded(e, [&](ptb::Engine &g) {
    g.set_output_name(filename ? filename : "fluxresult.vtk");
    return 0;
  });
}
int pumitally_set_option(pumitally_engine *e, const char *name, int64_t value) {
  return guarded(e, [&](ptb::Engine &g) { return g.set_option(name ? name : "", value); });
}

int64_t pumitally_get_option(const pumitally_engine *e, const char *name) {
  return (e && e->impl && name) ? e->impl->get_option(name) : -1;
}

int pumitally_copy_initial_position_device(pumitally_engine *e, const double *d_xyz, int32_t size,
                                           void *stream) {
  return guarded(e, [&](ptb::Engine &g) {
    return g.copy_initial_position_device(d_xyz, size, static_cast<cudaStream_t>(stream));
  });
}
int pumitally_move_to_next_location_device(pumitally_engine *e, const double *d_origin,
                                           const double *d_dest, const int8_t *d_flying,
                                           const double *d_weights, int32_t size, void *stream) {
  return guarded(e, [&](ptb::Engine &g) {
    return g.move_to_next_location_device(d_origin, d_dest, d_flying, d_weights, size,
                                          static_cast<cudaStream_t>(stream));
  });
}
int pumitally_set_state_device(pumitally_engine *e, const double *d_xyz, const int32_t *d_elem, int32_t first,
                               int32_t count, void *stream) {
  return guarded(e, [&](ptb::Engine &g) {
    return g.set_state_device(d_xyz, d_elem, first, count, static_cast<cudaStream_t>(stream));
  });
}
int pumitally_get_state_device(pumitally_engine *e, double *d_xyz, int32_t *d_elem, int32_t first, int32_t count,
                               void *stream) {
  return guarded(e, [&](ptb::Engine &g) {
    return g.get_state_device(d_xyz, d_elem, first, count, static_cast<cudaStream_t>(stream));
  });
}
int pumitally_get_flux_device(pumitally_engine *e, double *d_out, void *stream) {
  return guarded(e, [&](ptb::Engine &g) { return g.get_flux_device(d_out, static_cast<cudaStream_t>(stream)); });
}
double *pumitally_flux_device_ptr(pumitally_engine *e) {
  return (e && e->impl) ? e->impl->flux_device_ptr() : nullptr;
}
int pumitally_synchronize(pumitally_engine *e) {
  return guarded(e, [&](ptb::Engine &g) { return g.synchronize(); });
}

int pumitally_nccl_unique_id(uint8_t out_id[128]) { return ptb::nccl_get_unique_id(out_id); }
int pumitally_comm_init(pumitally_engine *e, int32_t rank, int32_t nranks, const uint8_t id[128]) {
  return guarded(e, [&](ptb::Engine &g) { return g.comm_init(rank, nranks, id); });
}
int pumitally_allreduce_tally(pumitally_engine *e) {
  return guarded(e, [&](ptb::Engine &g) { return g.allreduce_tally(); });
}
int pumitally_exchange_tally(pumitally_engine *e) {
  return guarded(e, [&](ptb::Engine &g) { return g.exchange_tally(); });
}
int pumitally_reduce_tally_to_owners(pumitally_engine *e) {
  return guarded(e, [&](ptb::Engine &g) { return g.reduce_tally_to_owners(); });
}

int pumitally_end_batch(pumitally_engine *e) {
  return guarded(e, [&](ptb::Engine &g) { return g.end_batch(); });
}
int pumitally_get_tally_statistics(pumitally_engine *e, double *out_mean, double *out_std_dev, int64_t n) {
  return guarded(e, [&](ptb::Engine &g) { return g.get_tally_statistics(out_mean, out_std_dev, n); });
}
int pumitally_get_max_relative_error(pumitally_engine *e, double threshold, double *out_max_rel, int64_t *out_index,
                                     int64_t *out_count_above) {
  return guarded(e, [&](ptb::Engine &g) {
    return g.max_relative_error(threshold, out_max_rel, out_index, out_count_above);
  });
}

int64_t pumitally_debug_order(pumitally_engine *e, int32_t *out, int64_t n) {
  if (!e || !e->impl) return -1;
  return e->impl->debug_order(out, n);
}

int64_t pumitally_debug_stage(const double *origin, const double *dest, int8_t *flying, const double *weights,
                              double *b_dest, double *b_w, int8_t *b_fly, int64_t n, int32_t compare,
                              int32_t threads, void *out_patches, int64_t cap) {
  try {
    ptb::HostStager st(threads, {});
    st.set_buffers(b_dest, b_w, b_fly);
    st.reserve(size_t(cap));
    st.begin(origin, dest, flying, weights, 0, n, compare != 0, static_cast<ptb::PatchEntry *>(out_patches));
    return st.end();
  } catch (const std::exception &ex) {
    fprintf(stderr, "[pumitally] ERROR: %s\n", ex.what());
    return -2;
  }
}

const char *pumitally_version(void) { return "pumitally-b200 0.2 (sm_100a)"; }

}  // extern "C"
