// Persistent-warp walk kernel (template) and its staging helpers, shared by the product
// translation unit (walk_kernels.cu: the kernels the engine actually chooses) and the
// experiments translation unit (experiments/walk_experiments.cu: measured alternatives that are
// not part of libpumitally.so).  Everything lives in an anonymous namespace: each TU gets its own
// instantiations.
#pragma once
#include <algorithm>
#include <cstddef>
#include <cstdint>

#include "walk_compact.cuh"
#include "walk_core.cuh"
#include "walk_kernels.hpp"

namespace ptb {
namespace {
__device__ __forceinline__ void flush_counters(const WalkParams &P, const Counters &c) {
  const unsigned segs = __reduce_add_sync(0xffffffffu, c.segs);
  const unsigned tracks = __reduce_add_sync(0xffffffffu, c.tracks);
  const unsigned relocs = __reduce_add_sync(0xffffffffu, c.relocs);
  const unsigned lost = __reduce_add_sync(0xffffffffu, c.lost);
  const unsigned fallbacks = __reduce_add_sync(0xffffffffu, c.fallbacks);
  if ((threadIdx.x & 31) == 0) {
    if (fallbacks) atomicAdd(&P.stats->fallbacks, (unsigned long long)fallbacks);
    if (segs) atomicAdd(&P.stats->segments, (unsigned long long)segs);
    if (tracks) atomicAdd(&P.stats->tracks, (unsigned long long)tracks);
    if (relocs) atomicAdd(&P.stats->relocations, (unsigned long long)relocs);
    if (lost) atomicAdd(&P.stats->lost, (unsigned long long)lost);
  }
}

__device__ __forceinline__ void load_face_256(const double *p, double &a, double &b, double &c,
                                              double &d) {
  asm volatile("ld.global.nc.v4.f64 {%0,%1,%2,%3}, [%4];" : "=d"(a), "=d"(b), "=d"(c), "=d"(d) : "l"(p));
}

constexpr int kRowBytes = 144;

__device__ __forceinline__ uint32_t smem_u32(const void *p) {
  return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_%=:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra DONE_%=;\n"
      "bra WAIT_%=;\n"
      "DONE_%=:\n"
      "}\n" ::"r"(bar),
      "r"(parity)
      : "memory");
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void *src, uint32_t bytes,
                                         uint32_t bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::
          "r"(dst),
      "l"(src), "r"(bytes), "r"(bar)
      : "memory");
}

// ---------------------------------------------------------------- variant 3
// Persistent warps with per-lane refill.  Track lengths are roughly geometric
// and relocation walks are ~10x longer than tally walks, so with one particle
// per thread a warp idles most of its lanes (measured: 3.9 of 32 lanes active
// per instruction).  Here every warp owns two shared-memory stages of 32
// particles each, filled asynchronously by the TMA unit (cp.async.bulk of the
// SoA/AoS slices, completion on an mbarrier); a lane that finishes its particle
// takes the next slot of the current stage in the same loop iteration, and
// chunks of 32 particles are claimed from a global counter so long walks never
// hold back the rest of the range.

constexpr int kChunk = 16;  // particles per staged chunk (all slice sizes stay multiples of 16 bytes)
constexpr uint32_t kB8 = 8u * kChunk, kB24 = 24u * kChunk, kB32 = 32u * kChunk, kB1 = 1u * kChunk;

struct __align__(64) ParticleStage {
  double origin[3 * kChunk];
  double dest[3 * kChunk];
  ParticleState state[kChunk];
  double w[kChunk];
  int8_t fly[kChunk];
  int32_t id[kChunk];  // gather mode: particle id of each slot
};
static_assert(sizeof(ParticleStage) >= kChunk * sizeof(PackedRow) && sizeof(ParticleStage) % 32 == 0 && offsetof(ParticleStage, state) % 32 == 0 && offsetof(ParticleStage, w) % 16 == 0 && offsetof(ParticleStage, fly) % 16 == 0, "stage layout");

__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}

__device__ __forceinline__ void stage_load(const WalkParams &P, int chunk, ParticleStage *st,
                                           uint32_t bar, int lane) {
  const long long base = (long long)P.begin + (long long)chunk * kChunk;
  const int count = (int)min((long long)kChunk, (long long)P.end - base);
  if (count == kChunk && P.bulk_ok) {
    if (lane == 0) {
      const uint32_t bytes = kB32 + (P.origin ? kB24 : 0u) + (P.dest ? kB24 + kB8 : 0u) +
                             (P.flying ? kB1 : 0u);
      mbar_expect_tx(bar, bytes);
      bulk_g2s(smem_u32(st->state), P.state + base, kB32, bar);
      if (P.origin) bulk_g2s(smem_u32(st->origin), P.origin + 3 * base, kB24, bar);
      if (P.dest) {
        bulk_g2s(smem_u32(st->dest), P.dest + 3 * base, kB24, bar);
        bulk_g2s(smem_u32(st->w), P.weights + base, kB8, bar);
      }
      if (P.flying) bulk_g2s(smem_u32(st->fly), P.flying + base, kB1, bar);
    }
  } else {
    // ragged last chunk, or caller pointers that are not 16-byte aligned
    if (lane < count) {
      const long long i = base + lane;
      st->state[lane] = load_state(P.state + i);
      if (P.origin)
        for (int k = 0; k < 3; ++k) st->origin[3 * lane + k] = P.origin[3 * i + k];
      if (P.dest) {
        for (int k = 0; k < 3; ++k) st->dest[3 * lane + k] = P.dest[3 * i + k];
        st->w[lane] = P.weights[i];
      }
      if (P.flying) st->fly[lane] = P.flying[i];
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(bar);
  }
}

// begin_particle() reading the staged copy instead of global memory
__device__ __forceinline__ void begin_from_stage(const WalkParams &P, const ParticleStage *st, int s,
                                                 Ray &r, Counters &c) {
  r.stage = kStageDone;
  const bool fly = P.flying ? (st->fly[s] == 1) : true;
  if (!fly) return;
  const double x = st->state[s].x, y = st->state[s].y, z = st->state[s].z;
  r.e = st->state[s].elem;
  if (P.origin) {
    const double tx = st->origin[3 * s], ty = st->origin[3 * s + 1], tz = st->origin[3 * s + 2];
    if (tx != x || ty != y || tz != z) {
      if (!all_finite(tx, ty, tz)) {  // unusable origin: the particle sits this move out
        c.lost++;
        return;
      }
      start_reloc(P, r, x, y, z, tx, ty, tz);
      return;
    }
  }
  if (P.dest) start_tally_to(P, r, x, y, z, st->dest[3 * s], st->dest[3 * s + 1], st->dest[3 * s + 2], st->w[s], c, true);
}

// begin_particle() for a packed row (only flying particles have rows).  Returns the particle id.
__device__ __forceinline__ int begin_from_row(const WalkParams &P, const PackedRow *row, Ray &r, Counters &c) {
  const int id = row->id;
  const uint32_t el = row->elem;
  const double ox = row->ox, oy = row->oy, oz = row->oz;
  if (el >> 31) {  // re-sourced: phase 1 from the stored position (rare)
    if (!all_finite(ox, oy, oz)) {  // unusable origin: the particle sits this move out
      c.lost++;
      return id;
    }
    const ParticleState s0 = load_state(P.state + id);
    r.e = s0.elem;
    start_reloc(P, r, s0.x, s0.y, s0.z, ox, oy, oz);
    return id;
  }
  r.e = (int32_t)(el & kIdMask);
  start_tally_to(P, r, ox, oy, oz, row->dx, row->dy, row->dz, row->w, c, true);
  return id;
}

// Fetch modes of the persistent kernel (how a lane gets its 128-byte tet record):
//   0  four plain 256-bit loads
//   1  as 0, tet loads carry an L2 evict_last policy and skip L1; the particle stream
//      (staging copies, state stores) is evict_first -- keeps the tet table L2-resident
//   2  as 1, plus the L2::128B prefetch size (first sector miss pulls the whole line)
//   3  one cp.async.bulk of 128 B per lane into a shared-memory row (policies as 1)
//   (4 was a cooperative quad-load + shared-memory transpose; measured 4.9 ms vs 3.0 ms on c2,
//      profiles/r01/README.md section c/d, and removed)
//   5  as 1 but the tet loads allocate in L1 (worth it once particles are processed in
//      spatial order and neighbouring lanes/warps revisit the same records)
//   6  compact layout + edge-function exit test (walk_compact.cuh): one 32-byte TetLinks sector and
//      one 32-byte vertex per crossing, both L2-resident; degenerate rays finish on the plane records
//   7, 8  as 1 and 5 with the warp-aggregated tally of walk_core.cuh (experiment)
//   9, 10 as 1 and 5 with the lean crossing step (plane_step_lean: the three record loads issued as one
//         block, payload decoded once, ray target re-read at the end of the ray instead of held in registers)
enum : int { kFetchPlain = 0, kFetchPolicy = 1, kFetchPolicy128 = 2, kFetchBulk = 3, kFetchPolicyL1 = 5, kFetchEdge = 6,
             kFetchPolicyAgg = 7, kFetchPolicyL1Agg = 8, kFetchLean = 9, kFetchLeanL1 = 10 };

__device__ __forceinline__ uint64_t l2_policy_keep() {
  uint64_t p;
  asm("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
  return p;
}
__device__ __forceinline__ uint64_t l2_policy_stream() {
  uint64_t p;
  asm("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
  return p;
}
// same value, created where it is used: keeps the policy out of the registers that stay live
// across the crossing loop of the compact-layout kernel
__device__ __forceinline__ uint64_t l2_policy_stream_now() {
  uint64_t p;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
  return p;
}
__device__ __forceinline__ void bulk_g2s_hint(uint32_t dst, const void *src, uint32_t bytes,
                                              uint32_t bar, uint64_t pol) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], "
      "%2, [%3], %4;" ::"r"(dst),
      "l"(src), "r"(bytes), "r"(bar), "l"(pol)
      : "memory");
}
template <int FETCH>
__device__ __forceinline__ void load_face(const double *p, uint64_t pol, double &a, double &b,
                                          double &c, double &d) {
  if constexpr (FETCH == kFetchPolicy || FETCH == kFetchPolicyAgg)
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.v4.f64 {%0,%1,%2,%3}, [%4], %5;"
        : "=d"(a), "=d"(b), "=d"(c), "=d"(d) : "l"(p), "l"(pol));
  else if constexpr (FETCH == kFetchPolicyL1 || FETCH == kFetchPolicyL1Agg)
    asm volatile("ld.global.nc.L2::cache_hint.v4.f64 {%0,%1,%2,%3}, [%4], %5;"
        : "=d"(a), "=d"(b), "=d"(c), "=d"(d) : "l"(p), "l"(pol));
  else if constexpr (FETCH == kFetchPolicy128)
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.L2::128B.v4.f64 {%0,%1,%2,%3}, [%4], %5;"
        : "=d"(a), "=d"(b), "=d"(c), "=d"(d) : "l"(p), "l"(pol));
  else
    load_face_256(p, a, b, c, d);
}

// stage_load() with an L2 policy on the streamed particle data
__device__ __forceinline__ void stage_load_hint(const WalkParams &P, int chunk, ParticleStage *st,
                                                uint32_t bar, int lane, uint64_t pol) {
  const long long base = (long long)P.begin + (long long)chunk * kChunk;
  const int count = (int)min((long long)kChunk, (long long)P.end - base);
  if (count == kChunk && P.bulk_ok) {
    if (lane == 0) {
      const uint32_t bytes = kB32 + (P.origin ? kB24 : 0u) + (P.dest ? kB24 + kB8 : 0u) +
                             (P.flying ? kB1 : 0u);
      mbar_expect_tx(bar, bytes);
      bulk_g2s_hint(smem_u32(st->state), P.state + base, kB32, bar, pol);
      if (P.origin) bulk_g2s_hint(smem_u32(st->origin), P.origin + 3 * base, kB24, bar, pol);
      if (P.dest) {
        bulk_g2s_hint(smem_u32(st->dest), P.dest + 3 * base, kB24, bar, pol);
        bulk_g2s_hint(smem_u32(st->w), P.weights + base, kB8, bar, pol);
      }
      if (P.flying) bulk_g2s_hint(smem_u32(st->fly), P.flying + base, kB1, bar, pol);
    }
  } else {
    stage_load(P, chunk, st, bar, lane);  // ragged / unaligned: plain path
  }
}

// ---- gather mode: the chunk's particles are not contiguous (order[] comes from the binning
// pass); every lane pulls its particle's fields with 8/4-byte cp.async copies that complete on
// the stage's mbarrier (cp.async.mbarrier.arrive.noinc: one arrival per lane, barrier count 32)
// (the gathered particle data is used once: evict_first keeps it from displacing tet records in L2)
__device__ __forceinline__ void cp_async_8(uint32_t dst, const void *src, uint64_t pol) {
  asm volatile("cp.async.ca.shared.global.L2::cache_hint [%0], [%1], 8, %2;" ::"r"(dst), "l"(src), "l"(pol)
               : "memory");
}
__device__ __forceinline__ void cp_async_16(uint32_t dst, const void *src, uint64_t pol) {
  asm volatile("cp.async.cg.shared.global.L2::cache_hint [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "l"(pol)
               : "memory");
}
__device__ __forceinline__ void cp_async_arrive_noinc(uint32_t bar) {
  asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(bar) : "memory");
}
// `id` = this lane's particle for the chunk (lanes >= count hold garbage and copy nothing)
__device__ __forceinline__ void stage_gather(const WalkParams &P, int id, int count, ParticleStage *st,
                                             uint32_t bar, int lane, uint64_t pol) {
  if (lane < count) {
    const int i = id;
    st->id[lane] = i;
    cp_async_16(smem_u32(&st->state[lane]), P.state + i, pol);
    cp_async_16(smem_u32(&st->state[lane]) + 16u, reinterpret_cast<const char *>(P.state + i) + 16, pol);
    if (P.origin) {
#pragma unroll
      for (int k = 0; k < 3; ++k)
        cp_async_8(smem_u32(&st->origin[3 * lane + k]), P.origin + 3 * (size_t)i + k, pol);
    }
    if (P.dest) {
#pragma unroll
      for (int k = 0; k < 3; ++k)
        cp_async_8(smem_u32(&st->dest[3 * lane + k]), P.dest + 3 * (size_t)i + k, pol);
      cp_async_8(smem_u32(&st->w[lane]), P.weights + i, pol);
    }
  }
  cp_async_arrive_noinc(bar);
}

// One crossing on the plane records.  Entry-face elision: after a crossing the face the ray came
// in through is known (r.entry) and can never be the exit, so only the other three 32-byte
// sectors of the record are fetched; the first tet of a ray needs all four.
template <int FETCH>
__device__ __forceinline__ void plane_step(const WalkParams &P, int my_i, Ray &r, Counters &c, uint64_t pol) {
  ExitScan sc;
  const double *rec = P.tets[r.e].d;
  const int en = r.entry;
  double q[3][4], q3[4];
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    const int fk = k + ((en >= 0 && k >= en) ? 1 : 0);
    load_face<FETCH>(rec + 4 * fk, pol, q[k][0], q[k][1], q[k][2], q[k][3]);
  }
  if (en < 0) load_face<FETCH>(rec + 12, pol, q3[0], q3[1], q3[2], q3[3]);
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    const int fk = k + ((en >= 0 && k >= en) ? 1 : 0);
    int32_t nb, bk;
    face_payload(q[k][0], q[k][1], q[k][2], q[k][3], r.e, fk, nb, bk);
    scan_face(sc, q[k][0], q[k][1], q[k][2], q[k][3], nb, bk, r.ox, r.oy, r.oz, r.ux, r.uy, r.uz);
  }
  if (en < 0) {
    int32_t nb, bk;
    face_payload(q3[0], q3[1], q3[2], q3[3], r.e, 3, nb, bk);
    scan_face(sc, q3[0], q3[1], q3[2], q3[3], nb, bk, r.ox, r.oy, r.oz, r.ux, r.uy, r.uz);
  }
  advance<false, FETCH == kFetchPolicyAgg || FETCH == kFetchPolicyL1Agg>(P, my_i, r, exit_parameter(sc), sc.nbr, sc.back, c, true);
}

// Lean crossing step.  ncu's source view of plane_step() (profiles/r02/README.md, section kernel) shows the
// compiler sinking the third record load below the arithmetic on the first two -- its latency is then
// paid a second time (14 % of all stall samples) -- and ~330 warp instructions per warp step.  Here the
// three loads are one asm block (issued back to back, before any use), the neighbour is decoded once,
// the parallel-face tolerance is computed once per step, and the ray target is not carried in registers
// (end_ray<true> re-reads it from the caller's array), which makes room for the loads in flight.
template <bool L1ALLOC>
__device__ __forceinline__ void load_faces3(const double *p0, const double *p1, const double *p2, uint64_t pol,
                                            double (&q)[3][4]) {
  if constexpr (L1ALLOC)
    asm volatile(
        "ld.global.nc.L2::cache_hint.v4.f64 {%0,%1,%2,%3}, [%12], %15;\n\t"
        "ld.global.nc.L2::cache_hint.v4.f64 {%4,%5,%6,%7}, [%13], %15;\n\t"
        "ld.global.nc.L2::cache_hint.v4.f64 {%8,%9,%10,%11}, [%14], %15;"
        : "=d"(q[0][0]), "=d"(q[0][1]), "=d"(q[0][2]), "=d"(q[0][3]), "=d"(q[1][0]), "=d"(q[1][1]), "=d"(q[1][2]),
          "=d"(q[1][3]), "=d"(q[2][0]), "=d"(q[2][1]), "=d"(q[2][2]), "=d"(q[2][3])
        : "l"(p0), "l"(p1), "l"(p2), "l"(pol));
  else
    asm volatile(
        "ld.global.nc.L1::no_allocate.L2::cache_hint.v4.f64 {%0,%1,%2,%3}, [%12], %15;\n\t"
        "ld.global.nc.L1::no_allocate.L2::cache_hint.v4.f64 {%4,%5,%6,%7}, [%13], %15;\n\t"
        "ld.global.nc.L1::no_allocate.L2::cache_hint.v4.f64 {%8,%9,%10,%11}, [%14], %15;"
        : "=d"(q[0][0]), "=d"(q[0][1]), "=d"(q[0][2]), "=d"(q[0][3]), "=d"(q[1][0]), "=d"(q[1][1]), "=d"(q[1][2]),
          "=d"(q[1][3]), "=d"(q[2][0]), "=d"(q[2][1]), "=d"(q[2][2]), "=d"(q[2][3])
        : "l"(p0), "l"(p1), "l"(p2), "l"(pol));
}

template <int FETCH>
__device__ __forceinline__ void plane_step_lean(const WalkParams &P, int my_i, Ray &r, Counters &c, uint64_t pol) {
  constexpr bool L1 = FETCH == kFetchLeanL1;
  const double *rec = P.tets[r.e].d;
  const int en = r.entry;
  // faces 0,1,2 with the entry face skipped: offsets (en<=0), (en<=1)+1, (en<=2)+2 for en >= 0; 0,1,2 for en < 0
  const int f0 = (en == 0) ? 1 : 0, f1 = (en >= 0 && en <= 1) ? 2 : 1, f2 = (en >= 0 && en <= 2) ? 3 : 2;
  double q[3][4], q3[4];
  load_faces3<L1>(rec + 4 * f0, rec + 4 * f1, rec + 4 * f2, pol, q);
  if (en < 0) load_face<L1 ? kFetchPolicyL1 : kFetchPolicy>(rec + 12, pol, q3[0], q3[1], q3[2], q3[3]);
  const double tol = kParallelTol * (fabs(r.ux) + fabs(r.uy) + fabs(r.uz));
  LeanScan sc;
  scan_face_lean(sc, q[0][0], q[0][1], q[0][2], q[0][3], f0, tol, r.ox, r.oy, r.oz, r.ux, r.uy, r.uz);
  scan_face_lean(sc, q[1][0], q[1][1], q[1][2], q[1][3], f1, tol, r.ox, r.oy, r.oz, r.ux, r.uy, r.uz);
  scan_face_lean(sc, q[2][0], q[2][1], q[2][2], q[2][3], f2, tol, r.ox, r.oy, r.oz, r.ux, r.uy, r.uz);
  if (en < 0) scan_face_lean(sc, q3[0], q3[1], q3[2], q3[3], 3, tol, r.ox, r.oy, r.oz, r.ux, r.uy, r.uz);
  int32_t nb, bk;
  decode_lean(sc, r.e, nb, bk);
  // The next tet is known here, ~80 instructions (a division, the tally, the loop overhead) before its
  // record is asked for: start the line on its way from DRAM to L2 now.  Half of the record fetches miss
  // in L2 on config c2 and a warp issues only one instruction every ~14 cycles, so the prefetch has
  // roughly a DRAM latency of head start.
  if (nb >= 0 && sc.bnum < sc.bden)
    asm volatile("prefetch.global.L2::evict_last [%0];" ::"l"(P.tets + nb));
  advance<true>(P, my_i, r, exit_parameter(sc), nb, bk, c, true);
}

// ---- compact layout (kFetchEdge) ----------------------------------------------------------
constexpr int kPlaneMode = -2;  // EdgeRay::dv of a ray that is finishing on the plane records

__device__ __forceinline__ void ld256_b64(const void *p, uint64_t pol, unsigned long long &a,
                                          unsigned long long &b, unsigned long long &c, unsigned long long &d) {
  asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.v4.b64 {%0,%1,%2,%3}, [%4], %5;"
               : "=l"(a), "=l"(b), "=l"(c), "=l"(d) : "l"(p), "l"(pol));
}

// First tet of a ray, out of line: its register footprint (four vertices, six edge functions)
// must not set the allocation of the per-crossing path.  The TetStart line has already been
// loaded by the caller (together with the other lanes' per-crossing loads, so the warp waits for
// memory once per iteration); everything crosses the call by value.
struct FirstOut {
  EdgeRay g;
  double texit;
  int32_t next, roles, ok;
};
__device__ __noinline__ FirstOut edge_first_compute(double v0, double v1, double v2, double v3, double v4, double v5,
                                                    double v6, double v7, double v8, double v9, double v10,
                                                    double v11, unsigned long long w0, unsigned long long w1,
                                                    unsigned long long w2, unsigned long long w3, double ox, double oy,
                                                    double oz, double ux, double uy, double uz) {
  const double v[12] = {v0, v1, v2, v3, v4, v5, v6, v7, v8, v9, v10, v11};
  TetLinks L;
  L.nbr[0] = (uint32_t)w0; L.nbr[1] = (uint32_t)(w0 >> 32); L.nbr[2] = (uint32_t)w1; L.nbr[3] = (uint32_t)(w1 >> 32);
  L.opp[0] = (uint32_t)w2; L.opp[1] = (uint32_t)(w2 >> 32); L.opp[2] = (uint32_t)w3; L.opp[3] = (uint32_t)(w3 >> 32);
  Ray r;
  r.ox = ox; r.oy = oy; r.oz = oz; r.ux = ux; r.uy = uy; r.uz = uz;
  FirstOut o;
  o.g.dv = 0;
  o.texit = 0.0;
  o.next = -1;
  o.roles = 0;
  o.ok = edge_first(r, o.g, L, v, o.texit, o.next, o.roles) ? 1 : 0;
  return o;
}

// A ray that met a coplanar edge finishes on the plane records.  Out of line and by value for the
// same reason as edge_first_step: rare, and its registers must not count against the crossing loop.
struct PlaneOut {
  double texit;
  int32_t next, back;
};
__device__ __noinline__ PlaneOut plane_fallback_step(const TetRecord *tets, int32_t e, int32_t en, double ox,
                                                     double oy, double oz, double ux, double uy, double uz) {
  const uint64_t pol = l2_policy_stream_now();
  ExitScan sc;
  const double *rec = tets[e].d;
#pragma unroll
  for (int f = 0; f < 4; ++f) {
    if (f == en) continue;
    double a, b, c, d;
    load_face<kFetchPolicy>(rec + 4 * f, pol, a, b, c, d);
    int32_t nb, bk;
    face_payload(a, b, c, d, e, f, nb, bk);
    scan_face(sc, a, b, c, d, nb, bk, ox, oy, oz, ux, uy, uz);
  }
  PlaneOut o;
  o.texit = exit_parameter(sc);
  o.next = sc.nbr;
  o.back = sc.back;
  return o;
}

// One crossing of the edge-function walk.  Requests first, for every lane at once: the TetLinks
// sector of the current tet + the one new vertex (keep policy; vertices also allocate in L1), or on
// the first tet of a ray the four sectors of its TetStart line (streaming policy).  `tgt` is the
// lane's shared-memory slot holding the ray's target (Ray::tx,ty,tz are not kept in registers).
__device__ __forceinline__ void edge_persist_step(const WalkParams &P, int my_i, Ray &r, EdgeRay &g,
                                                  Counters &c, uint64_t keep, double *tgt) {
  const bool plane = g.dv == kPlaneMode;
  const bool first = r.entry < 0;
  unsigned long long w0 = 0, w1 = 0, w2 = 0, w3 = 0;
  double v[12];
  if (!plane) {
    const TetStart *S = P.starts + r.e;
    const void *pa = first ? (const void *)&S->links : (const void *)(P.links + r.e);
    const double *pb = first ? S->v : reinterpret_cast<const double *>(P.verts + g.dv);
    const uint64_t pol = first ? l2_policy_stream_now() : keep;
    ld256_b64(pa, pol, w0, w1, w2, w3);
    load_face<kFetchPolicyL1>(pb, pol, v[0], v[1], v[2], v[3]);
    if (first) {
      load_face<kFetchPolicy>(S->v + 4, pol, v[4], v[5], v[6], v[7]);
      load_face<kFetchPolicy>(S->v + 8, pol, v[8], v[9], v[10], v[11]);
    }
  }
  double texit;
  int32_t next, roles;
  bool ok = true;
  if (plane) {
    const PlaneOut o = plane_fallback_step(P.tets, r.e, r.entry, r.ox, r.oy, r.oz, r.ux, r.uy, r.uz);
    texit = o.texit;
    next = o.next;
    roles = o.back;
  } else if (first) {
    const FirstOut o = edge_first_compute(v[0], v[1], v[2], v[3], v[4], v[5], v[6], v[7], v[8], v[9], v[10], v[11],
                                          w0, w1, w2, w3, r.ox, r.oy, r.oz, r.ux, r.uy, r.uz);
    g = o.g;
    texit = o.texit;
    next = o.next;
    roles = o.roles;
    ok = o.ok != 0;
  } else {
    TetLinks L;
    L.nbr[0] = (uint32_t)w0; L.nbr[1] = (uint32_t)(w0 >> 32); L.nbr[2] = (uint32_t)w1; L.nbr[3] = (uint32_t)(w1 >> 32);
    L.opp[0] = (uint32_t)w2; L.opp[1] = (uint32_t)(w2 >> 32); L.opp[2] = (uint32_t)w3; L.opp[3] = (uint32_t)(w3 >> 32);
    ok = edge_step(r, g, L, v[0], v[1], v[2], texit, next, roles);
  }
  if (ok) {
    // the ray ends in this step (reached / hull / iteration limit): end_ray() needs its target
    if (!(texit < 1.0) || next < 0 || r.iters + 1 >= P.max_iters) {
      r.tx = tgt[0]; r.ty = tgt[1]; r.tz = tgt[2];
    }
    advance(P, my_i, r, texit, next, roles, c, true);
    if (r.iters == 0 && r.stage != kStageDone) {  // a new ray (phase 2 after phase 1)
      tgt[0] = r.tx; tgt[1] = r.ty; tgt[2] = r.tz;
      if (plane) g.dv = 0;  // it starts on the fast path again
    }
  } else {  // coplanar edge: redo this tet, and the rest of the ray, with the planes
    g.dv = kPlaneMode;
    r.entry = -1;
    atomicAdd(&P.stats->fallbacks, 1ull);
  }
}

constexpr int kClaimRun = 4;  // gather mode: a warp takes up to this many consecutive chunks per ticket

// REFILL_T: idle lanes are topped up only when at least this many have finished -- the
// refill code then runs with REFILL_T+ active lanes instead of the ~3 that finish per
// iteration, at the price of a few idle lanes in the walk step.
// STAGING: 0 = particle arrays streamed in storage order (TMA bulk copies of the SoA/AoS slices),
// 1 = gather through order[] (binned), 2 = packed rows written by the binning pass (binned, streamed).
template <int BLOCK, int FETCH, int MINB, int REFILL_T, int STAGING>
__global__ void __launch_bounds__(BLOCK, MINB) walk_persist_kernel(const WalkParams P) {
  constexpr bool GATHER = STAGING == 1;
  constexpr bool PACKED = STAGING == 2;
  constexpr int WARPS = BLOCK / 32;
  constexpr bool kBulkTets = FETCH == kFetchBulk;
  constexpr bool kRows = FETCH == kFetchBulk;
  __shared__ ParticleStage stages[WARPS][2];
  __shared__ __align__(8) unsigned long long bars[WARPS][3];
  __shared__ __align__(128) unsigned char rows[kRows ? WARPS : 1][kRows ? 32 * kRowBytes : 16];
  constexpr bool kEdge = FETCH == kFetchEdge;
  __shared__ double targets[kEdge ? BLOCK : 1][3];  // compact layout: each lane's ray target
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const uint32_t bar0 = smem_u32(&bars[warp][0]);
  const uint32_t bar_row = bar0 + 16;
  const uint32_t row = smem_u32(&rows[kRows ? warp : 0][kRows ? lane * kRowBytes : 0]);
  if (lane == 0) {
    mbar_init(bar0, GATHER ? 32 : 1);
    mbar_init(bar0 + 8, GATHER ? 32 : 1);
    mbar_init(bar_row, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }
  __syncwarp();
  const uint64_t keep = FETCH != kFetchPlain ? l2_policy_keep() : 0;
  const uint64_t strm = (FETCH == kFetchEdge) ? 0 : ((FETCH != kFetchPlain || GATHER) ? l2_policy_stream() : 0);
  const int total = (GATHER || PACKED) ? (int)__ldg(P.work_count) : P.end - P.begin;
  const int nchunks = (total + kChunk - 1) / kChunk;
  // Gather mode: a ticket is a run of kClaimRun chunks = 64 particles whose ids sit in two
  // registers per lane.  The *next* ticket is claimed, and its ids requested, one run ahead, so
  // neither the atomic nor the id loads are ever waited for.
  static_assert(kClaimRun * kChunk == 64, "two id registers per lane cover the largest ticket");
  const int claim_run = GATHER ? min(max(P.claim_run, 1), kClaimRun) : 1;
  int run_base = 0, run_next = 0, run_end = 0, ids0 = 0, ids1 = 0;
  int pend_base = -1, pend0 = 0, pend1 = 0;
  // next ticket of `run` chunks: its first chunk, or a value >= nchunks when nothing is left (warp-uniform)
  auto take = [&](int run) -> int {
    int c = 0;
    if (lane == 0) c = (int)atomicAdd(P.work_counter, (unsigned)run);
    return __shfl_sync(0xffffffffu, c, 0);
  };
  auto fetch_ticket = [&]() {
    pend_base = take(claim_run);
    const long long p0 = (long long)pend_base * kChunk + lane, p1 = p0 + 32;
    const long long pe = min((long long)total, ((long long)pend_base + claim_run) * kChunk);
    pend0 = p0 < pe ? __ldg(P.order + p0) : 0;
    pend1 = p1 < pe ? __ldg(P.order + p1) : 0;
  };
  auto load_stage = [&](int chunk, ParticleStage *st, uint32_t bar) {
    if constexpr (PACKED) {
      // one bulk copy: the chunk's rows are contiguous and every row is 64 bytes, ragged tail included
      if (lane == 0) {
        const uint32_t bytes = 64u * (uint32_t)min(kChunk, total - chunk * kChunk);
        mbar_expect_tx(bar, bytes);
        bulk_g2s_hint(smem_u32(st), P.rows + (size_t)chunk * kChunk, bytes, bar, strm);
      }
    } else if constexpr (GATHER) {
      const int k = chunk - run_base;  // chunk's position in the current ticket (warp-uniform)
      const int id = __shfl_sync(0xffffffffu, (k >> 1) ? ids1 : ids0, ((k & 1) << 4) | (lane & 15));
      stage_gather(P, id, min(kChunk, total - chunk * kChunk), st, bar, lane,
                   FETCH == kFetchEdge ? l2_policy_stream_now() : strm);
    } else if constexpr (FETCH == kFetchPlain) {
      stage_load(P, chunk, st, bar, lane);
    } else {
      stage_load_hint(P, chunk, st, bar, lane, FETCH == kFetchEdge ? l2_policy_stream_now() : strm);
    }
  };
  auto claim = [&]() -> int {
    int c = 0;
    if constexpr (GATHER) {
      if (run_next >= run_end) {
        if (pend_base < 0) fetch_ticket();
        run_base = run_next = pend_base;
        run_end = pend_base + claim_run;
        ids0 = pend0;
        ids1 = pend1;
        fetch_ticket();
      }
      c = run_next++;
    } else {
      c = take(1);
    }
    return c < nchunks ? c : -1;
  };

  int cur = 0, cursor = 0, cur_count = 0;
  uint32_t parity = 0;  // bit b = phase parity of barrier b (0,1 particle stages; 2 tet rows)
  int chunk_cur = claim();
  if (chunk_cur >= 0) load_stage(chunk_cur, &stages[warp][0], bar0);
  int chunk_next = chunk_cur >= 0 ? claim() : -1;
  if (chunk_next >= 0) load_stage(chunk_next, &stages[warp][1], bar0 + 8);
  if (chunk_cur >= 0) {
    mbar_wait(bar0, 0);
    parity ^= 1u;
    cur_count = min(kChunk, total - chunk_cur * kChunk);
  }

  Counters c;
  Ray r;
  EdgeRay g;  // only live in the compact-layout instantiation
  g.dv = 0;
  r.stage = kStageDone;
  int my_i = 0;
  for (;;) {
    unsigned idle = __ballot_sync(0xffffffffu, r.stage == kStageDone);
    while (cur_count > 0 && (int)__popc(idle) >= REFILL_T) {
      const int slot = cursor + __popc(idle & ((1u << lane) - 1u));
      if (r.stage == kStageDone && slot < cur_count) {
        if constexpr (PACKED) {
          my_i = begin_from_row(P, reinterpret_cast<const PackedRow *>(&stages[warp][cur]) + slot, r, c);
        } else {
          my_i = GATHER ? stages[warp][cur].id[slot] : P.begin + chunk_cur * kChunk + slot;
          begin_from_stage(P, &stages[warp][cur], slot, r, c);
        }
        if constexpr (FETCH == kFetchEdge) {
          g.dv = 0;
          if (r.stage != kStageDone) {
            targets[threadIdx.x][0] = r.tx; targets[threadIdx.x][1] = r.ty; targets[threadIdx.x][2] = r.tz;
          }
        }
      }
      __syncwarp();
      cursor += __popc(idle);
      if (cursor >= cur_count) {
        // every slot of this stage has been handed out: recycle it for the chunk after next
        const int recycled = cur;
        chunk_cur = chunk_next;
        cur ^= 1;
        cursor = 0;
        cur_count = 0;
        chunk_next = -1;
        if (chunk_cur >= 0) {
          mbar_wait(bar0 + 8 * cur, (parity >> cur) & 1u);
          parity ^= 1u << cur;
          cur_count = min(kChunk, total - chunk_cur * kChunk);
          chunk_next = claim();
          if (chunk_next >= 0) {
            if (lane == 0) asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            load_stage(chunk_next, &stages[warp][recycled], bar0 + 8 * recycled);
          }
        }
      }
      idle = __ballot_sync(0xffffffffu, r.stage == kStageDone);
    }
    if (idle == 0xffffffffu) break;  // no lane active and nothing left to hand out
    if constexpr (kBulkTets) {
      const unsigned act = ~idle;
      if (lane == __ffs(act) - 1) mbar_expect_tx(bar_row, 128u * __popc(act));
      if (r.stage != kStageDone) bulk_g2s_hint(row, P.tets + r.e, 128u, bar_row, keep);
      mbar_wait(bar_row, (parity >> 2) & 1u);
      parity ^= 4u;
    }
    if (r.stage != kStageDone) {
      if constexpr (FETCH == kFetchEdge) {
        edge_persist_step(P, my_i, r, g, c, keep, &targets[kEdge ? threadIdx.x : 0][0]);
      } else if constexpr (kRows) {
        ExitScan sc;
        double raw[16];
#pragma unroll
        for (int j = 0; j < 8; ++j)
          asm volatile("ld.shared.v2.f64 {%0,%1}, [%2];"
                       : "=d"(raw[2 * j]), "=d"(raw[2 * j + 1])
                       : "r"(row + 16 * j));
        scan_record(raw, r.e, r.ox, r.oy, r.oz, r.ux, r.uy, r.uz, sc);
        advance(P, my_i, r, exit_parameter(sc), sc.nbr, sc.back, c, true);
      } else if constexpr (FETCH == kFetchLean || FETCH == kFetchLeanL1) {
        plane_step_lean<FETCH>(P, my_i, r, c, keep);
      } else {
        plane_step<FETCH>(P, my_i, r, c, keep);
      }
    }
  }
  flush_counters(P, c);
}

template <int BLOCK, int FETCH, int MINB, int REFILL_T = 1, int GATHER = 0, int CARVE = -1>
cudaError_t launch_persist(const WalkParams &p, long long n, cudaStream_t stream) {
  static int sms = 0, occ = 0;
  if (!sms) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    // leave as much of the unified L1/smem array to shared memory as the kernel can use
    cudaFuncSetAttribute(walk_persist_kernel<BLOCK, FETCH, MINB, REFILL_T, GATHER>,
                         cudaFuncAttributePreferredSharedMemoryCarveout,
                         CARVE < 0 ? (int)cudaSharedmemCarveoutMaxShared : CARVE);
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, walk_persist_kernel<BLOCK, FETCH, MINB, REFILL_T, GATHER>, BLOCK, 0);
    if (occ < 1) occ = 1;
  }
  const long long nchunks = (n + kChunk - 1) / kChunk;
  const long long want = (nchunks + BLOCK / 32 - 1) / (BLOCK / 32);
  const unsigned grid = (unsigned)std::min<long long>(want, (long long)sms * occ);
  cudaError_t e = cudaMemsetAsync(p.work_counter, 0, sizeof(unsigned int), stream);
  if (e != cudaSuccess) return e;
  walk_persist_kernel<BLOCK, FETCH, MINB, REFILL_T, GATHER><<<grid, BLOCK, 0, stream>>>(p);
  return cudaGetLastError();
}

}  // namespace
}  // namespace ptb
