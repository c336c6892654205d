// Worker pool + stage pass of the host-pointer path (see host_stage.hpp).
#include "host_stage.hpp"

#include <immintrin.h>
#include <sched.h>
#include <sys/syscall.h>
#include <unistd.h>

#include <algorithm>
#include <cctype>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <sstream>

namespace ptb {

// ------------------------------------------------------------------------------------ pool

namespace {
constexpr int kSpinsBeforeSleep = 4000;  // ~200 us of _mm_pause on current x86 parts

void pin_to(const std::vector<int> &cpus) {
  if (cpus.empty()) return;
  cpu_set_t set;
  CPU_ZERO(&set);
  for (int c : cpus)
    if (c >= 0 && c < CPU_SETSIZE) CPU_SET(c, &set);
  sched_setaffinity(0, sizeof(set), &set);  // best effort
}
}  // namespace

HostPool::HostPool(int nthreads, const std::vector<int> &cpus) : n_(std::max(1, nthreads)) {
  for (int t = 0; t < n_; ++t)
    threads_.emplace_back([this, t, cpus] {
      pin_to(cpus);
      worker(t);
    });
}

HostPool::~HostPool() {
  if (in_flight_) end();
  {
    std::lock_guard<std::mutex> lk(m_);
    stop_.store(true);
    gen_.fetch_add(1);
  }
  cv_.notify_all();
  for (auto &t : threads_) t.join();
}

void HostPool::worker(int tid) {
  uint64_t seen = 0;
  for (;;) {
    int spins = 0;
    while (gen_.load(std::memory_order_acquire) == seen) {
      if (++spins < kSpinsBeforeSleep) {
        _mm_pause();
        continue;
      }
      std::unique_lock<std::mutex> lk(m_);
      sleepers_.fetch_add(1);
      cv_.wait(lk, [&] { return gen_.load(std::memory_order_acquire) != seen; });
      sleepers_.fetch_sub(1);
    }
    if (stop_.load()) return;
    seen = gen_.load(std::memory_order_acquire);
    (*job_)(tid);
    if (done_.fetch_add(1, std::memory_order_acq_rel) + 1 == n_) {
      // last one out wakes the caller if it went to sleep in end()
      std::lock_guard<std::mutex> lk(done_m_);
      done_cv_.notify_one();
    }
  }
}

void HostPool::begin(const std::function<void(int)> &fn) {
  if (in_flight_) end();
  job_ = &fn;
  done_.store(0, std::memory_order_relaxed);
  {
    std::lock_guard<std::mutex> lk(m_);  // pairs with the predicate check of a worker going to sleep
    gen_.fetch_add(1, std::memory_order_release);
  }
  if (sleepers_.load() > 0) cv_.notify_all();
  in_flight_ = true;
}

// The caller must not spin for the length of a job: a spinning thread on the sibling hyperthread of a
// worker halves that worker's speed, and the slowest worker sets the pace (measured: 2x on the whole
// pass).  A short spin catches jobs that are about to finish, then it sleeps until the last worker
// signals.
void HostPool::end() {
  if (!in_flight_) return;
  for (int spins = 0; spins < 200 && done_.load(std::memory_order_acquire) != n_; ++spins) _mm_pause();
  if (done_.load(std::memory_order_acquire) != n_) {
    std::unique_lock<std::mutex> lk(done_m_);
    done_cv_.wait(lk, [&] { return done_.load(std::memory_order_acquire) == n_; });
  }
  in_flight_ = false;
}

void HostPool::repin(const std::vector<int> &cpus) {
  if (cpus.empty()) return;
  run([&](int) { pin_to(cpus); });
}

void HostPool::barrier() {
  if (n_ == 1) return;
  const uint64_t g = bar_gen_.load(std::memory_order_acquire);
  if (bar_count_.fetch_add(1, std::memory_order_acq_rel) + 1 == n_) {
    bar_count_.store(0, std::memory_order_relaxed);
    bar_gen_.fetch_add(1, std::memory_order_release);
  } else {
    while (bar_gen_.load(std::memory_order_acquire) == g) _mm_pause();
  }
}

// ------------------------------------------------------------------------- sizing / placement

namespace {

int env_int(const char *name, int dflt) {
  const char *v = std::getenv(name);
  return (v && *v) ? std::atoi(v) : dflt;
}

// "0-3,8,10-11" -> {0,1,2,3,8,10,11}
std::vector<int> parse_cpulist(const std::string &s) {
  std::vector<int> out;
  std::stringstream ss(s);
  std::string tok;
  while (std::getline(ss, tok, ',')) {
    int a = 0, b = 0;
    if (sscanf(tok.c_str(), "%d-%d", &a, &b) == 2) {
      for (int c = a; c <= b && c < 4096; ++c) out.push_back(c);
    } else if (sscanf(tok.c_str(), "%d", &a) == 1) {
      out.push_back(a);
    }
  }
  return out;
}

double cgroup_cpu_quota() {
  {  // cgroup v2
    std::ifstream f("/sys/fs/cgroup/cpu.max");
    std::string q;
    double period = 0;
    if (f >> q >> period && q != "max" && period > 0) return std::atof(q.c_str()) / period;
  }
  {  // cgroup v1
    std::ifstream fq("/sys/fs/cgroup/cpu/cpu.cfs_quota_us"), fp("/sys/fs/cgroup/cpu/cpu.cfs_period_us");
    double q = 0, p = 0;
    if (fq >> q && fp >> p && q > 0 && p > 0) return q / p;
  }
  return 1e9;
}

}  // namespace

int default_host_threads() {
  const int forced = env_int("PUMITALLY_HOST_THREADS", 0);
  if (forced > 0) return std::min(forced, 256);
  // this rank's share of the machine (hardware threads and CPU quota divided by the ranks on the node),
  // but never more than its own affinity mask offers (a rank bound to its GPU's NUMA node shares that
  // node only with the ranks of the node's other GPUs, so the mask itself is not divided)
  cpu_set_t set;
  const int hw = std::max(1, int(std::thread::hardware_concurrency()));
  int avail = hw;
  if (sched_getaffinity(0, sizeof(set), &set) == 0) avail = CPU_COUNT(&set);
  int local = env_int("LOCAL_WORLD_SIZE", 0);
  if (local <= 0) local = env_int("OMPI_COMM_WORLD_LOCAL_SIZE", 0);
  if (local <= 0) local = env_int("SLURM_NTASKS_PER_NODE", 0);
  if (local <= 0) local = 1;
  const double n = std::min({double(avail), cgroup_cpu_quota() / local, double(hw) / local});
  return std::max(1, std::min(32, int(n + 0.5)));
}

std::vector<int> gpu_local_cpus(const std::string &pci_bus_id) {
  if (env_int("PUMITALLY_HOST_PIN", 1) == 0) return {};
  std::string id = pci_bus_id;
  for (auto &c : id) c = char(std::tolower((unsigned char)c));
  std::ifstream f("/sys/bus/pci/devices/" + id + "/local_cpulist");
  std::string line;
  if (!f || !std::getline(f, line)) return {};
  std::vector<int> local = parse_cpulist(line), out;
  cpu_set_t set;
  if (sched_getaffinity(0, sizeof(set), &set) != 0) return {};
  for (int c : local)
    if (c < CPU_SETSIZE && CPU_ISSET(c, &set)) out.push_back(c);
  // a node that offers fewer CPUs than the mask as a whole is not worth confining the pool to
  if (int(out.size()) * 4 < CPU_COUNT(&set)) return {};
  return out;
}

namespace {
std::vector<int> in_affinity_mask(const std::vector<int> &cpus) {
  std::vector<int> out;
  cpu_set_t set;
  if (sched_getaffinity(0, sizeof(set), &set) != 0) return out;
  for (int c : cpus)
    if (c >= 0 && c < CPU_SETSIZE && CPU_ISSET(c, &set)) out.push_back(c);
  return out;
}
}  // namespace

int numa_node_of(const void *p, size_t bytes) {
  const int forced = env_int("PUMITALLY_HOST_NODE", -1);
  if (forced >= 0) return forced;
  if (!p || bytes == 0) return -1;
  constexpr int kSamples = 16;
  const long page = sysconf(_SC_PAGESIZE);
  void *pages[kSamples];
  int status[kSamples];
  const uintptr_t base = reinterpret_cast<uintptr_t>(p) & ~uintptr_t(page - 1);
  for (int k = 0; k < kSamples; ++k) {
    pages[k] = reinterpret_cast<void *>(base + ((bytes / kSamples * size_t(k)) & ~size_t(page - 1)));
    status[k] = -1;
  }
  if (syscall(SYS_move_pages, 0, (unsigned long)kSamples, pages, nullptr, status, 0) != 0) return -1;
  int votes[64] = {0}, best = -1;
  for (int k = 0; k < kSamples; ++k)
    if (status[k] >= 0 && status[k] < 64) ++votes[status[k]];
  for (int n = 0; n < 64; ++n)
    if (votes[n] > 0 && (best < 0 || votes[n] > votes[best])) best = n;
  return best;
}

std::vector<int> numa_node_cpus(int node) {
  if (node < 0 || env_int("PUMITALLY_HOST_PIN", 1) == 0) return {};
  std::ifstream f("/sys/devices/system/node/node" + std::to_string(node) + "/cpulist");
  std::string line;
  if (!f || !std::getline(f, line)) return {};
  return in_affinity_mask(parse_cpulist(line));
}

// -------------------------------------------------------------------------------- stage pass

namespace {

inline bool differs(const double *a, const double *b) {
  uint64_t x[3], y[3];
  std::memcpy(x, a, 24);
  std::memcpy(y, b, 24);
  return ((x[0] ^ y[0]) | (x[1] ^ y[1]) | (x[2] ^ y[2])) != 0;
}

// one particle, plain stores
// a changed origin: recorded while there is room; past that the list is void (np keeps counting so
// that the caller sees np > cap) but the staging goes on
inline void record(const double *o, int64_t i, PatchEntry *patches, int64_t &np, int64_t cap) {
  if (np < cap) patches[np] = PatchEntry{o[0], o[1], o[2], int32_t(i), 0};
  ++np;
}

inline void stage_one(const double *origin, const double *dest, const double *weights, double *b_dest, double *b_w,
                      int64_t i, bool compare, PatchEntry *patches, int64_t &np, int64_t cap) {
  if (compare && differs(origin + 3 * i, b_dest + 3 * i)) record(origin + 3 * i, i, patches, np, cap);
  b_dest[3 * i] = dest[3 * i];
  b_dest[3 * i + 1] = dest[3 * i + 1];
  b_dest[3 * i + 2] = dest[3 * i + 2];
  b_w[i] = weights[i];
}

int64_t stage_scalar(const double *origin, const double *dest, int8_t *flying, const double *weights, double *b_dest,
                     double *b_w, int8_t *b_fly, int64_t lo, int64_t hi, bool compare, PatchEntry *patches,
                     int64_t cap) {
  int64_t np = 0;
  for (int64_t i = lo; i < hi; ++i) {
    const int8_t f = flying[i];
    b_fly[i] = f;
    flying[i] = 0;
    stage_one(origin, dest, weights, b_dest, b_w, i, compare && f == 1, patches, np, cap);
  }
  return np <= cap ? np : -1;
}

// Blocked version: 256 particles at a time (origin + mirror + dest + weights of a block = 20 KB, L1
// resident), one simple two-stream pass after the other inside the block -- (1) compare origin with
// the mirror, (2) dest -> mirror slots, (3) weights, (4) flying.  Interleaving all seven streams in
// one loop runs at half the speed (measured): the hardware prefetchers and the fill buffers do
// best on few streams at a time.  The mirror lines are still in L1 from pass 1 when pass 2
// overwrites them, so plain stores are right (a non-temporal store would first evict the line).
// Slots of non-flying particles are refilled too (branch-free copy); an origin is only reported
// when the particle flies.
constexpr int64_t kBlock = 256;

__attribute__((target("avx2"))) void copy_block(double *dst, const double *src, int64_t doubles) {
  int64_t k = 0;
  for (; k + 8 <= doubles; k += 8) {
    const __m256i a = _mm256_loadu_si256((const __m256i *)(src + k)), b = _mm256_loadu_si256((const __m256i *)(src + k + 4));
    _mm256_storeu_si256((__m256i *)(dst + k), a);
    _mm256_storeu_si256((__m256i *)(dst + k + 4), b);
  }
  for (; k < doubles; ++k) dst[k] = src[k];
}

__attribute__((target("avx2"))) int64_t stage_avx2(const double *origin, const double *dest, int8_t *flying,
                                                   const double *weights, double *b_dest, double *b_w, int8_t *b_fly,
                                                   int64_t lo, int64_t hi, bool compare, PatchEntry *patches,
                                                   int64_t cap) {
  int64_t np = 0;
  for (int64_t b0 = lo; b0 < hi; b0 += kBlock) {
    const int64_t b1 = std::min(hi, b0 + kBlock), cnt = b1 - b0;
    if (compare) {
      const double *o = origin + 3 * b0;
      const double *m = b_dest + 3 * b0;
      int64_t g = 0;
      for (; g + 4 <= cnt; g += 4) {  // 4 particles = 96 bytes = three 256-bit lanes
        const double *og = o + 3 * g, *mg = m + 3 * g;
        const __m256i x0 = _mm256_xor_si256(_mm256_loadu_si256((const __m256i *)og), _mm256_loadu_si256((const __m256i *)mg));
        const __m256i x1 = _mm256_xor_si256(_mm256_loadu_si256((const __m256i *)(og + 4)), _mm256_loadu_si256((const __m256i *)(mg + 4)));
        const __m256i x2 = _mm256_xor_si256(_mm256_loadu_si256((const __m256i *)(og + 8)), _mm256_loadu_si256((const __m256i *)(mg + 8)));
        const __m256i x = _mm256_or_si256(_mm256_or_si256(x0, x1), x2);
        if (!_mm256_testz_si256(x, x)) {
          for (int k = 0; k < 4; ++k)
            if (flying[b0 + g + k] == 1 && differs(og + 3 * k, mg + 3 * k)) record(og + 3 * k, b0 + g + k, patches, np, cap);
        }
      }
      for (; g < cnt; ++g)
        if (flying[b0 + g] == 1 && differs(o + 3 * g, m + 3 * g)) record(o + 3 * g, b0 + g, patches, np, cap);
    }
    copy_block(b_dest + 3 * b0, dest + 3 * b0, 3 * cnt);
    if (cnt == kBlock && (reinterpret_cast<uintptr_t>(b_w + b0) & 63u) == 0) {
      // the weight slots are written only: whole 64-byte lines with non-temporal stores, no
      // read-for-ownership (the dest slots above were just read by the compare pass)
      for (int64_t k = 0; k < kBlock; k += 8) {
        const __m256i a = _mm256_loadu_si256((const __m256i *)(weights + b0 + k)), b = _mm256_loadu_si256((const __m256i *)(weights + b0 + k + 4));
        _mm256_stream_si256((__m256i *)(b_w + b0 + k), a);
        _mm256_stream_si256((__m256i *)(b_w + b0 + k + 4), b);
      }
    } else {
      copy_block(b_w + b0, weights + b0, cnt);
    }
    std::memcpy(b_fly + b0, flying + b0, size_t(cnt));
    std::memset(flying + b0, 0, size_t(cnt));
  }
  _mm_sfence();
  return np <= cap ? np : -1;
}

}  // namespace

int64_t stage_range(const double *origin, const double *dest, int8_t *flying, const double *weights,
                    double *b_dest, double *b_w, int8_t *b_fly, int64_t lo, int64_t hi, bool compare,
                    PatchEntry *patches, int64_t cap) {
  static const bool have_avx2 = __builtin_cpu_supports("avx2");
  static const bool force_scalar = std::getenv("PUMITALLY_STAGE_SCALAR") != nullptr;
  if (have_avx2 && !force_scalar)
    return stage_avx2(origin, dest, flying, weights, b_dest, b_w, b_fly, lo, hi, compare, patches, cap);
  return stage_scalar(origin, dest, flying, weights, b_dest, b_w, b_fly, lo, hi, compare, patches, cap);
}

// ------------------------------------------------------------------------------- stager

void HostStager::reserve(size_t cap) {
  if (cap == cap_ && !tls_.empty()) return;
  cap_ = cap;
  const size_t T = size_t(pool_.size());
  // blocks are claimed dynamically, so a worker may collect more than its even share of a chunk's
  // entries; beyond four times that the chunk counts as overflowed (its origins then travel whole)
  tls_cap_ = std::min(cap, 4 * (cap / T)) + 64;
  tls_.assign(T, std::vector<PatchEntry>());
  for (auto &v : tls_) v.resize(tls_cap_);
  counts_.assign(T, 0);
}

void HostStager::begin(const double *origin, const double *dest, int8_t *flying, const double *weights,
                       int64_t b, int64_t e, bool compare, PatchEntry *out) {
  job_ = Job{origin, dest, weights, flying, b, e, compare, out, 0};
  next_block_.store(0, std::memory_order_relaxed);
  pool_.begin(fn_);
}

int64_t HostStager::end() {
  pool_.end();
  return job_.total;
}

void HostStager::work(int t) {
  Job &j = job_;
  const int T = pool_.size();
  // Blocks of kGrain particles are claimed from a shared counter: the pace is set by the slowest
  // worker (one that shares a core with another busy thread runs at half speed), so the split must
  // not be fixed in advance.
  PatchEntry *mine = tls_[size_t(t)].data();
  int64_t np = 0;
  bool overflow = false;
  for (;;) {
    const int64_t blk = next_block_.fetch_add(1, std::memory_order_relaxed);
    const int64_t lo = j.b + blk * kGrain;
    if (lo >= j.e) break;
    const int64_t hi = std::min(j.e, lo + kGrain);
    const int64_t c = stage_range(j.origin, j.dest, j.flying, j.weights, b_dest_, b_w_, b_fly_, lo, hi, j.compare,
                                  mine + np, int64_t(tls_cap_) - np);
    if (c < 0) overflow = true;
    else np += c;
  }
  counts_[size_t(t)] = overflow ? -1 : np;
  if (!j.compare) return;
  pool_.barrier();
  int64_t off = 0, all = 0;
  bool any_overflow = false;
  for (int k = 0; k < T; ++k) {
    const int64_t ck = counts_[size_t(k)];
    any_overflow |= ck < 0;
    if (k < t) off += ck;
    all += ck;
  }
  if (any_overflow || all > int64_t(cap_)) {
    if (t == 0) j.total = -1;
    return;
  }
  if (np > 0) std::memcpy(j.out + off, mine, size_t(np) * sizeof(PatchEntry));
  if (t == 0) j.total = all;
}

}  // namespace ptb
