// A stand-in for the OpenMC event loop that drives the tally library through the same four
// call sites the OpenMC fork uses (reference: images/public_methods_explanation.svg, README.md:136-149):
//
//   openmc_init                      -> PumiTally(mesh, n, argc, argv)
//   process_init_events              -> CopyInitialPosition(source positions)
//   process_advance_particle_events  -> MoveToNextLocation(origin, dest, flying, weights)   (per event sweep)
//   openmc_simulation_finalize       -> WriteTallyResults()
//
// Physics is a toy: isotropic flights with exponential lengths inside a box; a particle that leaks is
// "absorbed" and re-sampled at a new source site, which is what exercises the relocate-to-origin phase.
// Only <pumitally/PumiTally.h> and -lpumitally are needed for the reference's four calls; the optional
// batches / per-source normalisation below (what the reference leaves as TODOs, PumiTallyImpl.h:170-171)
// use the additive <pumitally/PumiTallyExtras.h>.
//
//   g++ -std=c++17 -I include examples/openmc_like_driver.cpp -L pumiumtally_b200/lib -lpumitally \
//       -Wl,-rpath,$PWD/pumiumtally_b200/lib -o driver && ./driver box:20,20,20 1000000 20 [inactive_batches [energy_groups [active_batches]]]
//
// energy_groups > 1 turns the tally into a filtered one (pumitally::SetScoreBins): each flight scores into the
// flux array of the group it was sampled in; the VTK output then carries flux_bin<k> next to flux (their sum).
// active_batches > 1 runs that many active batches of `sweeps` sweeps and closes each with pumitally::EndBatch:
// the VTK output then holds the mean over the batches with its standard deviation (flux_std_dev), and the
// driver prints the largest relative error of the tally (pumitally::MaxRelativeError, OpenMC's tally trigger).
#include <chrono>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <string>
#include <vector>

#include "pumitally/PumiTally.h"
#include "pumitally/PumiTallyExtras.h"

namespace {
struct Rng {  // SplitMix64
  uint64_t s;
  double next() {
    uint64_t z = (s += 0x9E3779B97F4A7C15ull);
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return double((z ^ (z >> 31)) >> 11) * 0x1.0p-53;
  }
};
}  // namespace

int main(int argc, char **argv) {
  const std::string mesh = argc > 1 ? argv[1] : "box:20,20,20";
  const int n = argc > 2 ? std::atoi(argv[2]) : 100000;
  const int sweeps = argc > 3 ? std::atoi(argv[3]) : 10;
  const int inactive = argc > 4 ? std::atoi(argv[4]) : 0;  // batches of `sweeps` sweeps run and discarded first
  const int groups = argc > 5 ? std::atoi(argv[5]) : 1;    // energy groups of the score filter
  const int active = argc > 6 ? std::atoi(argv[6]) : 1;    // active batches, each closed by EndBatch when > 1
  double box[3] = {20, 20, 20};
  if (mesh.rfind("box:", 0) == 0) std::sscanf(mesh.c_str() + 4, "%lf,%lf,%lf", &box[0], &box[1], &box[2]);

  pumitally::PumiTally tally(mesh, n, argc, argv);  // openmc_init

  Rng rng{0x5EED};
  std::vector<double> pos(3 * size_t(n)), origin(3 * size_t(n)), dest(3 * size_t(n)), weight(n, 1.0);
  std::vector<int8_t> flying(n, 1);
  std::vector<int32_t> group(n, 0);
  if (groups > 1 && pumitally::SetScoreBins(tally, groups)) return 1;
  auto sample_site = [&](double *p) {
    for (int d = 0; d < 3; ++d) p[d] = (1e-6 + (1 - 2e-6) * rng.next()) * box[d];
  };
  for (int i = 0; i < n; ++i) sample_site(&pos[3 * size_t(i)]);
  tally.CopyInitialPosition(pos.data(), 3 * n);  // process_init_events

  // per-source-particle normalisation: divide the normalised flux by the total weight of the batch's first tracks
  if (inactive > 0) pumitally::SetSourceNormalization(tally, 3);
  const auto t0 = std::chrono::steady_clock::now();
  long long flights = 0, leaks = 0;
  const int batches = inactive + (active > 1 ? active : 1);
  for (int batch = 0; batch < batches; ++batch) {
  if (batch > 0 && batch <= inactive) {  // an inactive batch ends: discard its tally, keep the particles where they are
    pumitally::ResetTally(tally);
    flights = leaks = 0;
  }
  for (int s = 0; s < sweeps; ++s) {  // process_advance_particle_events
    for (int i = 0; i < n; ++i) {
      double *p = &pos[3 * size_t(i)], *o = &origin[3 * size_t(i)], *d = &dest[3 * size_t(i)];
      for (int k = 0; k < 3; ++k) o[k] = p[k];
      const double mu = 2 * rng.next() - 1, phi = 6.283185307179586 * rng.next();
      const double len = -3.0 * std::log(1.0 - rng.next()), st = std::sqrt(1 - mu * mu);
      d[0] = o[0] + len * st * std::cos(phi);
      d[1] = o[1] + len * st * std::sin(phi);
      d[2] = o[2] + len * mu;
      flying[i] = 1;
      weight[i] = 0.5 + 0.5 * rng.next();
      if (groups > 1) group[i] = int32_t(rng.next() * groups);  // the "energy" after the last collision
      bool inside = true;
      for (int k = 0; k < 3; ++k) inside = inside && d[k] >= 0 && d[k] <= box[k];
      if (inside) { for (int k = 0; k < 3; ++k) p[k] = d[k]; }
      else { sample_site(p); ++leaks; }  // leaked: next flight starts at a fresh source site
      ++flights;
    }
    if (groups > 1)
      pumitally::MoveToNextLocationBinned(tally, origin.data(), dest.data(), flying.data(), weight.data(), group.data(), 3 * n);
    else
      tally.MoveToNextLocation(origin.data(), dest.data(), flying.data(), weight.data(), 3 * n);
  }
  if (active > 1 && batch >= inactive && pumitally::EndBatch(tally)) return 1;  // an active batch ends
  }
  const double secs = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
  tally.WriteTallyResults();  // openmc_simulation_finalize
  std::printf("DRIVER_OK %lld flights (%lld leaked and re-sampled) in %d sweeps, %.3f s host loop + tally calls, "
              "source normalisation %.6f\n",
              flights, leaks, sweeps, secs, pumitally_get_source_normalization(pumitally::engine_of(tally)));
  if (active > 1) {
    double max_rel = 0.0;
    int64_t where = -1, above = 0;
    if (pumitally::MaxRelativeError(tally, 0.05, &max_rel, &where, &above)) return 1;
    std::printf("TALLY_TRIGGER %d active batches: max relative error %.17g at %lld, %lld bins above 0.05\n", active,
                max_rel, (long long)where, (long long)above);
  }
  return 0;
}
