// Host side of the host-pointer MoveToNextLocation path: a private worker pool and the per-chunk
// "stage" pass that turns the caller's (pageable) arrays into what actually has to cross PCIe.
//
// The reference copies origin, dest, flying and weights to the device with blocking deep_copies
// (PumiTallyImpl.cpp:159-193, 223-236): 57 bytes per particle per move.  A transport code's next
// origin is, for every particle that was not re-sourced, bit for bit the destination it passed in
// the previous call, and the device still holds those destinations.  So the engine keeps a pinned,
// per-particle copy of the previous dest/weight/flying arrays -- which is at the same time the DMA
// source of this move (no second copy) and the mirror the next origin array is compared against --
// and uploads only dest + weight + flying plus a short list of origins that really changed
// (32 + ~2 bytes per particle instead of 57).  The pass runs on a small pool of threads pinned to
// the GPU's NUMA node, chunk by chunk, while the previous chunk is on the wire.
#pragma once
#include <atomic>
#include <condition_variable>
#include <cstdint>
#include <functional>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "walk_core.cuh"  // PatchEntry

namespace ptb {

// Fork-join pool of n worker threads (the caller is not one of them: while the workers stage chunk
// k+1 the caller enqueues the copies and kernels of chunk k).  Workers spin briefly for the next job
// (jobs of one move follow each other within tens of microseconds) and then sleep on a condition
// variable, so an idle engine burns no CPU.  One job in flight at a time; not re-entrant.
class HostPool {
 public:
  // cpus: logical CPUs the workers may run on (empty = leave the affinity alone)
  HostPool(int nthreads, const std::vector<int> &cpus);
  ~HostPool();
  HostPool(const HostPool &) = delete;
  HostPool &operator=(const HostPool &) = delete;
  int size() const { return n_; }
  // fn(worker id) on every worker; fn must stay alive until end() has returned
  void begin(const std::function<void(int)> &fn);
  void end();
  void run(const std::function<void(int)> &fn) { begin(fn); end(); }
  void barrier();  // for use inside fn: all n workers meet here
  // move the workers to another set of CPUs (they re-pin themselves; empty = no change)
  void repin(const std::vector<int> &cpus);

 private:
  void worker(int tid);
  int n_;
  std::vector<std::thread> threads_;
  std::mutex m_;
  std::condition_variable cv_;
  std::atomic<uint64_t> gen_{0};
  std::atomic<int> done_{0};
  std::atomic<int> sleepers_{0};
  std::atomic<bool> stop_{false};
  bool in_flight_ = false;
  const std::function<void(int)> *job_ = nullptr;
  std::atomic<int> bar_count_{0};
  std::atomic<uint64_t> bar_gen_{0};
  std::mutex done_m_;
  std::condition_variable done_cv_;
};

// How many workers the pool should have: PUMITALLY_HOST_THREADS if set, otherwise
// min(CPUs in the affinity mask, cgroup CPU quota) / ranks on this node (LOCAL_WORLD_SIZE,
// OMPI_COMM_WORLD_LOCAL_SIZE), clamped to [1, 32].
int default_host_threads();
// CPUs local to the PCI device (sysfs local_cpulist) that are also in the process's affinity mask;
// empty when unknown or when PUMITALLY_HOST_PIN=0.
std::vector<int> gpu_local_cpus(const std::string &pci_bus_id);
// NUMA node that holds most of the sampled pages of [p, p + bytes) (move_pages query; -1 = unknown,
// e.g. pages not touched yet), and the CPUs of a node that are in the process's affinity mask.
// The stage pass is a streaming read of the caller's arrays: per-thread throughput drops 2-4x when
// those reads cross the socket interconnect, so the workers run where the caller's memory is.
int numa_node_of(const void *p, size_t bytes);
std::vector<int> numa_node_cpus(int node);

// What one worker does with its share [lo, hi) of a chunk.  For every particle:
//   - if compare and flying[i] == 1 and origin[i] != mirror dest[i] bitwise -> PatchEntry appended
//   - b_dest[i] <- dest[i], b_w[i] <- weights[i], b_fly[i] <- flying[i]
//   - flying[i] <- 0 (PumiTallyImpl.cpp:169-172)
// b_dest doubles as the mirror: it still holds the previous move's destinations when it is read.
// (Slots of non-flying particles are refilled as well -- a branch-free copy is cheaper than
// skipping them; if the caller's dest of such a particle is not where the particle is, its next
// flight merely reports its origin as changed, and the device decides exactly as always.)
// Returns the number of patch entries written, or -1 if they did not fit in `cap` (the range is
// staged completely either way).
int64_t stage_range(const double *origin, const double *dest, int8_t *flying, const double *weights,
                    double *b_dest, double *b_w, int8_t *b_fly, int64_t lo, int64_t hi, bool compare,
                    PatchEntry *patches, int64_t cap);


// One chunk of a move at a time: the pool's workers split particles [b, e), run stage_range on their
// shares with private patch lists and pack those into `out`.  begin() returns at once; end() waits
// and gives the list length, or -1 when it exceeds `cap` (the chunk's origins are then sent whole).
class HostStager {
 public:
  HostStager(int nthreads, const std::vector<int> &cpus) : pool_(nthreads, cpus) {
    fn_ = [this](int t) { work(t); };
  }
  int threads() const { return pool_.size(); }
  HostPool &pool() { return pool_; }
  void set_buffers(double *b_dest, double *b_w, int8_t *b_fly) {
    b_dest_ = b_dest; b_w_ = b_w; b_fly_ = b_fly;
  }
  void reserve(size_t cap);  // largest list a chunk may produce
  void begin(const double *origin, const double *dest, int8_t *flying, const double *weights, int64_t b,
             int64_t e, bool compare, PatchEntry *out);
  int64_t end();

 private:
  void work(int t);
  HostPool pool_;
  std::function<void(int)> fn_;
  double *b_dest_ = nullptr, *b_w_ = nullptr;
  int8_t *b_fly_ = nullptr;
  static constexpr int64_t kGrain = 2048;  // particles per claimed block (multiple of the pass's 256-particle tile)
  std::atomic<int64_t> next_block_{0};
  size_t cap_ = 0, tls_cap_ = 0;
  std::vector<std::vector<PatchEntry>> tls_;
  std::vector<int64_t> counts_;
  struct Job {
    const double *origin, *dest, *weights;
    int8_t *flying;
    int64_t b, e;
    bool compare;
    PatchEntry *out;
    int64_t total;
  } job_{};
};

}  // namespace ptb
