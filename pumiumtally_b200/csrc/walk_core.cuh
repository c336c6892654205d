// Per-tet step of the adjacency walk: decode a packed TetRecord, find the exit
// face of the ray, decide reached / crossed / left-the-hull.
//
// This is the arithmetic the reference delegates to the external pumi-pic
// tracer (call site PumiTallyImpl.cpp:454; contract PumiTallyImpl.h:74-85)
// fused with the reference's own per-iteration functor
// (PumiTallyImpl.cpp:297-316): tally the piece inside the current tet
// (EvaluateFlux :352-380), clip at the hull (ApplyVacuumBC :256-286), advance
// (UpdateCurrentElement :243-254).  prev_xpoint (:322-350) is the register
// `tcur`.
//
// The functions are __host__ __device__ only so that tests/ can compile them
// with g++ and check the logic on a machine without a GPU; the library never
// runs them on the host.
#pragma once
#include <cstdint>

#if defined(__CUDACC__)
#define PTB_HD __host__ __device__ __forceinline__
#if defined(__CUDA_ARCH__)
#define PTB_UNROLL _Pragma("unroll")
#else
#define PTB_UNROLL  // nvcc's host pass hands the pragma to g++, which does not know it
#endif
#else
#define PTB_HD inline
#define PTB_UNROLL
#include <cmath>
#include <cstring>
#endif

#if defined(__CUDA_ARCH__)
#define PTB_LDG(p) __ldg(p)
// RED.E.ADD.F64 (Kokkos::atomic_add, Impl.cpp:376) carrying the same L2 evict_last priority as
// the tet records: with the default priority the (small, extremely hot) flux lines are the first
// victims of the evict_last tet stream and every second reduction misses in L2.
__device__ __forceinline__ void tally_add(double *ptr, double v) {
  unsigned long long pol;
  asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
  asm volatile("red.global.add.L2::cache_hint.f64 [%0], %1, %2;" ::"l"(ptr), "d"(v), "l"(pol) : "memory");
}
#define PTB_TALLY_ADD(ptr, v) tally_add((ptr), (v))
// Experiment (north_star: "warp-aggregated atomicAdd to cut contention"): lanes of the warp that tally
// into the same tet in this step are found with match.any, their contributions are summed with
// shuffles and one lane issues the reduction.  Called by every converged lane; `on` = this lane has
// something to add.  Measured in profiles/r02 (variants 28, 29); not used by the product kernels.
__device__ __forceinline__ void tally_add_aggregated(double *flux, int32_t e, double v, bool on) {
  const unsigned act = __activemask();
  const int lane = threadIdx.x & 31;
  unsigned peers = __match_any_sync(act, on ? e : -1 - lane);  // lanes with nothing to add match only themselves
  const int leader = __ffs(peers) - 1;
  double sum = 0.0;
  unsigned m = peers;
  while (__any_sync(act, m != 0)) {
    const int src = m ? __ffs(m) - 1 : lane;
    const double x = __shfl_sync(act, v, src);
    if (m) { sum += x; m &= m - 1; }
  }
  if (on && lane == leader) tally_add(flux + e, sum);
}
#else
#define PTB_LDG(p) (*(p))
#define PTB_TALLY_ADD(ptr, v) (*(ptr) += (v))  // test-only host build is single threaded
#endif

namespace ptb {

// low/high 32-bit halves of a double, portable between nvcc device code and g++
PTB_HD uint32_t dlo(double x) {
#if defined(__CUDA_ARCH__)
  return (uint32_t)__double2loint(x);
#else
  uint64_t u; memcpy(&u, &x, 8); return (uint32_t)u;
#endif
}
// Tet ids are 30-bit; the all-ones id marks the hull.
constexpr uint32_t kIdMask = 0x3fffffffu;

// byte 0 of four words -> one word (b0 | b1<<8 | b2<<16 | b3<<24)
PTB_HD uint32_t pack_low_bytes(uint32_t w0, uint32_t w1, uint32_t w2, uint32_t w3) {
#if defined(__CUDA_ARCH__)
  return __byte_perm(__byte_perm(w0, w1, 0x0040), __byte_perm(w2, w3, 0x0040), 0x5410);
#else
  return (w0 & 0xffu) | ((w1 & 0xffu) << 8) | ((w2 & 0xffu) << 16) | ((w3 & 0xffu) << 24);
#endif
}

// Payload of one face of tet `self` (the four doubles a,b,c,d of local face f): the id of the
// neighbour across it (-1 = hull) and `back`, the neighbour's local index of the shared face.
// Stored symmetrically -- bits 0..29 = self XOR neighbour, bits 30..31 = f XOR back -- so the
// payload, and with it the plane, is bit-identical in the two records that share the face.
PTB_HD void face_payload(double a, double b, double c, double d, int32_t self, int f, int32_t &nbr,
                         int32_t &back) {
  const uint32_t pay = pack_low_bytes(dlo(a), dlo(b), dlo(c), dlo(d));
  const uint32_t x = (pay ^ (uint32_t)self) & kIdMask;
  nbr = (int32_t)((x + 1u) & kIdMask) - 1;  // kIdMask -> -1 (hull), everything else unchanged
  back = (int32_t)((pay >> 30) ^ (uint32_t)f);
}

// Running minimum of the exit parameter over the faces scanned so far.  Ray x(t) = o + t*u,
// t in [0,1]; a face is a candidate when the ray leaves through it (n.u > 0).  Numerator and
// denominator depend only on the plane and the ray, never on the tet, so both tets sharing a
// face compute the identical quotient.  The minimum is selected by cross-multiplication
// (num_a*den_b < num_b*den_a, both den > 0): one fp64 division per crossing instead of one per
// face; ties within rounding pick either face, which only reorders a zero-length piece.
constexpr double kParallelTol = 1e-12;

struct ExitScan {
  double bnum = 1.0, bden = 0.0;  // t = +inf
  int32_t nbr = -2, back = -1;
};

PTB_HD void scan_face(ExitScan &s, double nx, double ny, double nz, double c, int32_t nbr,
                      int32_t back, double ox, double oy, double oz, double ux, double uy,
                      double uz) {
  const double den = nx * ux + ny * uy + nz * uz;
  const double num = c - (nx * ox + ny * oy + nz * oz);
  // A face counts as an exit candidate only if the ray leaves through it at a real angle:
  // n.u > kParallelTol*|u|_1, not n.u > 0.  (a) A plane component that is exactly zero carries the
  // payload byte as a denormal, so a ray exactly parallel to the face would see n.u = +-1e-321*|u|.
  // (b) A ray that runs inside a face plane or along a mesh edge sees n.u = rounding noise for the faces
  // that contain it, and num/den of such a face is an arbitrary number that can win the minimum.  No ray
  // that is not parallel to the face within 1e-12 rad is affected.
  const bool take = (den > kParallelTol * (fabs(ux) + fabs(uy) + fabs(uz))) && (num * s.bden < s.bnum * den);
  s.bnum = take ? num : s.bnum;
  s.bden = take ? den : s.bden;
  s.nbr = take ? nbr : s.nbr;
  s.back = take ? back : s.back;
}

// Lean flavour of the scan: instead of decoding the neighbour of every face and selecting among the
// decoded values, the raw payload word and the face index of the best face are kept and decoded once
// after the last face (6 integer instructions per face less).  Same selection rule, same result.
struct LeanScan {
  double bnum = 1.0, bden = 0.0;  // t = +inf
  uint32_t pay = 0;
  int32_t f = -1;  // -1: no exit candidate yet
};

PTB_HD void scan_face_lean(LeanScan &s, double nx, double ny, double nz, double c, int f, double tol, double ox,
                           double oy, double oz, double ux, double uy, double uz) {
  const double den = nx * ux + ny * uy + nz * uz;
  const double num = c - (nx * ox + ny * oy + nz * oz);
  const bool take = (den > tol) && (num * s.bden < s.bnum * den);  // tol = kParallelTol * |u|_1, see scan_face()
  const uint32_t pay = pack_low_bytes(dlo(nx), dlo(ny), dlo(nz), dlo(c));
  s.bnum = take ? num : s.bnum;
  s.bden = take ? den : s.bden;
  s.pay = take ? pay : s.pay;
  s.f = take ? f : s.f;
}

PTB_HD void decode_lean(const LeanScan &s, int32_t self, int32_t &nbr, int32_t &back) {
  const uint32_t x = (s.pay ^ (uint32_t)self) & kIdMask;
  nbr = s.f < 0 ? -2 : (int32_t)((x + 1u) & kIdMask) - 1;
  back = s.f < 0 ? -1 : (int32_t)((s.pay >> 30) ^ (uint32_t)s.f);
}

// bnum >= bden  <=>  t >= 1: the destination lies in this tet, no division needed
PTB_HD double exit_parameter(const ExitScan &s) {
  return (s.bnum < s.bden) ? s.bnum / s.bden : __builtin_huge_val();
}
PTB_HD double exit_parameter(const LeanScan &s) {
  return (s.bnum < s.bden) ? s.bnum / s.bden : __builtin_huge_val();
}

// All four faces of a record held as 16 raw doubles (variants that fetch the whole line).
PTB_HD void scan_record(const double (&r)[16], int32_t self, double ox, double oy, double oz,
                        double ux, double uy, double uz, ExitScan &s) {
PTB_UNROLL
  for (int f = 0; f < 4; ++f) {
    int32_t nb, bk;
    face_payload(r[4 * f], r[4 * f + 1], r[4 * f + 2], r[4 * f + 3], self, f, nb, bk);
    scan_face(s, r[4 * f], r[4 * f + 1], r[4 * f + 2], r[4 * f + 3], nb, bk, ox, oy, oz, ux, uy, uz);
  }
}


// ---------------------------------------------------------------------------
// Per-ray state machine shared by every kernel variant.
// ---------------------------------------------------------------------------

struct DeviceStats {
  unsigned long long segments;     // tally contributions (weighted phase, flying particles)
  unsigned long long tracks;       // flying particles in weighted phases
  unsigned long long relocations;  // crossings walked with tallying off
  unsigned long long lost;         // walks stopped by the iteration limit
  unsigned long long fallbacks;    // compact layout: rays handed to the plane records (coplanar edge)
};

struct TetRecord;
struct TetLinks;
struct VertexRec;
struct TetStart;

// Persistent per-particle state: position + parent element in one 32-byte, 32-byte aligned
// record = one DRAM/L2 sector.  A particle is read with one 256-bit load and written back with
// one full-sector 256-bit store (no read-modify-write fill), in whatever order particles are
// processed.  (Reference: DPS members origin + the tracer's elem_ids, PumiTallyImpl.h:39-41.)
struct alignas(32) ParticleState {
  double x, y, z;
  int32_t elem;
  int32_t pad;
};
static_assert(sizeof(ParticleState) == 32, "ParticleState must be one sector");

PTB_HD ParticleState load_state(const ParticleState *p) {
#if defined(__CUDA_ARCH__)
  unsigned long long a, b, c, d;
  asm volatile("ld.global.L1::no_allocate.v4.b64 {%0,%1,%2,%3}, [%4];" : "=l"(a), "=l"(b), "=l"(c), "=l"(d) : "l"(p));
  ParticleState s;
  s.x = __longlong_as_double((long long)a);
  s.y = __longlong_as_double((long long)b);
  s.z = __longlong_as_double((long long)c);
  s.elem = (int32_t)(d & 0xffffffffull);
  s.pad = 0;
  return s;
#else
  return *p;
#endif
}
PTB_HD void store_state(ParticleState *p, double x, double y, double z, int32_t elem) {
#if defined(__CUDA_ARCH__)
  asm volatile("st.global.L1::no_allocate.v4.b64 [%0], {%1,%2,%3,%4};" ::"l"(p),
               "l"((unsigned long long)__double_as_longlong(x)), "l"((unsigned long long)__double_as_longlong(y)),
               "l"((unsigned long long)__double_as_longlong(z)), "l"((unsigned long long)(uint32_t)elem)
               : "memory");
#else
  p->x = x; p->y = y; p->z = z; p->elem = elem; p->pad = 0;
#endif
}

// Uniform background grid over the mesh bounding box: cell -> the tet that
// contains the cell centre (-1 if the centre is outside the mesh).  A far
// relocation (re-sampled particle, initial localisation) starts its tally-off
// walk at the centre of the target's cell instead of at the particle's old
// position.  For a target inside the mesh both walks end in the tet that
// contains it, so the result is the reference's; if the seeded walk meets the
// hull the kernel falls back to the reference walk from the old position,
// which also reproduces the clip point of an out-of-mesh target.
struct SeedGrid {
  const int32_t *cell_tet;  // [nx*ny*nz]; nullptr = grid disabled
  const int32_t *cell_rank; // [nx*ny*nz] position of the cell along a Morton curve (binning key)
  double x0, y0, z0;        // low corner of the bounding box
  double h, inv_h;          // cell edge and its reciprocal
  double far2;              // seed only when |target - position|^2 exceeds this
  int32_t nx, ny, nz;
};

// Seed point of cell (cx,cy,cz): deliberately off-centre so that structured
// meshes whose cell centres lie on tet faces/edges do not start every seeded
// walk in a degenerate position.  Explicit fma: identical on host and device.
PTB_HD void seed_point(const SeedGrid &g, int cx, int cy, int cz, double &x, double &y, double &z) {
  x = fma(cx + 0.41421356237, g.h, g.x0);
  y = fma(cy + 0.57735026919, g.h, g.y0);
  z = fma(cz + 0.31830988618, g.h, g.z0);
}

// One entry of the origin patch list (host-pointer path, delta upload): particle idx starts this
// move at (x,y,z) instead of at the previous move's destination.  32 bytes = one sector.
struct alignas(32) PatchEntry {
  double x, y, z;
  int32_t idx;
  int32_t pad;
};

// One row of the packed, spatially sorted particle batch (variant "packed"): everything a flying
// particle needs for this move in one 64-byte line, written by the binning pass in cell order and
// streamed by the walk kernel with one bulk copy per chunk.  The stored position is not carried:
// for every continuing particle it equals `origin` bit for bit; the others (bit 31 of `elem` set)
// read their ParticleState when they start.
struct alignas(64) PackedRow {
  double ox, oy, oz;  // origin (= position before the move unless the relocate bit is set)
  double dx, dy, dz;  // destination
  double w;
  int32_t id;         // particle index in the caller's arrays
  uint32_t elem;      // bits 0..29 parent element, bit 31: origin differs from the stored position
};
static_assert(sizeof(PackedRow) == 64, "PackedRow must be one 64-byte line");

// One launch = one particle range of one MoveToNextLocation / CopyInitialPosition.
struct WalkParams {
  const TetRecord *tets;   // [E] packed records
  const TetLinks *links;   // [E] compact layout (walk_compact.cuh); nullptr when not uploaded
  const VertexRec *verts;  // [V]
  const TetStart *starts;  // [E]
  double *flux;            // [E] raw tally
  ParticleState *state;    // [N] persistent particle position + parent element
  const double *origin;    // [3N] AoS relocation target (phase 1), nullptr = skip phase
  const double *dest;      // [3N] AoS flight target (phase 2), nullptr = skip phase
  const int8_t *flying;    // [N], nullptr = every particle flies (localisation)
  const double *weights;   // [N]
  int32_t begin, end;      // particle range
  int32_t max_iters;       // crossing limit per walk ("May need more loops in search")
  int32_t bulk_ok;         // all particle arrays 16-byte aligned: cp.async.bulk staging allowed
  unsigned int *work_counter;  // chunk ticket of the persistent kernel (zeroed per launch)
  const int32_t *order;        // gather mode: ids of the flying particles in processing order
  const unsigned int *work_count;  // gather mode: number of entries in order[] (device scalar)
  int32_t claim_run;           // gather mode: chunks per ticket (1, 2 or 4)
  const PackedRow *rows;       // packed mode: work_count rows in processing order
  DeviceStats *stats;
  SeedGrid grid;
  double cx, cy, cz;           // mesh centre: the planes are stored relative to it (tet_mesh.hpp)
};

constexpr int kStageReloc = 0;  // phase 1: move to caller's origin, tally off
constexpr int kStageTally = 1;  // phase 2: fly to destination, tally on
constexpr int kStageDone = 2;
constexpr int kStageSeed = 3;   // phase 1 started from a seed-grid cell centre

struct Ray {
  double ox, oy, oz;  // ray origin (fixed for the whole walk), in mesh-centred coordinates
  double ux, uy, uz;  // target - origin
  double tx, ty, tz;  // target (stored exactly as given: it becomes the position when reached)
  double tcur;        // parameter of the last crossing (the reference's prev_xpoint)
  double wl;          // weight * |u|  (tally phase)
  int32_t e;          // current tet
  int32_t entry;      // local face of `e` the ray came in through (-1 at the start of a ray):
                      // it can never be the exit, so its sector need not be fetched
  int32_t stage;
  int32_t iters;
};

struct Counters {
  unsigned segs = 0, tracks = 0, relocs = 0, lost = 0, fallbacks = 0;
};

// (x,y,z) and the target are the caller's (absolute) coordinates; only the ray origin is translated,
// once: the direction is a difference and the target is kept as given (it becomes the stored position)
PTB_HD void set_ray(const WalkParams &P, Ray &r, double x, double y, double z, double tx, double ty, double tz) {
  r.ox = x - P.cx; r.oy = y - P.cy; r.oz = z - P.cz;
  r.ux = tx - x; r.uy = ty - y; r.uz = tz - z;
  r.tx = tx; r.ty = ty; r.tz = tz;
  r.tcur = 0.0;
  r.iters = 0;
  r.entry = -1;
}

// NaN or infinity in the caller's numbers must not reach the tally or the stored state: x*0 is 0 for
// every finite x and NaN otherwise.
PTB_HD bool all_finite(double a, double b, double c) { return (a * 0.0 + b * 0.0 + c * 0.0) == 0.0; }

// Tally phase towards (tx,ty,tz) with weight w.  A non-finite destination or weight turns the flight
// into a zero-length one (the particle stays where it is, nothing is tallied) and counts as lost.
PTB_HD void start_tally_to(const WalkParams &P, Ray &r, double x, double y, double z, double tx, double ty,
                           double tz, double w, Counters &c, bool writer) {
  if (!all_finite(tx, ty, tz) || !all_finite(w, 0.0, 0.0)) {
    tx = x; ty = y; tz = z;
    w = 0.0;
    if (writer) c.lost++;
  }
  set_ray(P, r, x, y, z, tx, ty, tz);
  const double len = sqrt(r.ux * r.ux + r.uy * r.uy + r.uz * r.uz);
  r.wl = w * len;
  r.stage = kStageTally;
  if (writer) c.tracks++;
}

PTB_HD void start_tally(const WalkParams &P, int i, Ray &r, double x, double y, double z,
                        Counters &c, bool writer) {
  start_tally_to(P, r, x, y, z, PTB_LDG(P.dest + 3 * (size_t)i), PTB_LDG(P.dest + 3 * (size_t)i + 1),
                 PTB_LDG(P.dest + 3 * (size_t)i + 2), PTB_LDG(P.weights + i), c, writer);
}

// Phase 1 for a particle at (x,y,z) in tet r.e whose caller-side origin is (tx,ty,tz).
PTB_HD void start_reloc(const WalkParams &P, Ray &r, double x, double y, double z, double tx,
                        double ty, double tz) {
  r.wl = 0.0;  // p_wgt = 0 during relocation (Impl.cpp:105)
  const SeedGrid &g = P.grid;
  if (g.cell_tet) {
    const double dx = tx - x, dy = ty - y, dz = tz - z;
    const double fx = (tx - g.x0) * g.inv_h, fy = (ty - g.y0) * g.inv_h, fz = (tz - g.z0) * g.inv_h;
    if (dx * dx + dy * dy + dz * dz > g.far2 && fx >= 0.0 && fy >= 0.0 && fz >= 0.0 &&
        fx < (double)g.nx && fy < (double)g.ny && fz < (double)g.nz) {
      const int cx = (int)fx, cy = (int)fy, cz = (int)fz;
      const int32_t seed = PTB_LDG(g.cell_tet + ((size_t)cz * g.ny + cy) * g.nx + cx);
      if (seed >= 0) {
        double sx, sy, sz;
        seed_point(g, cx, cy, cz, sx, sy, sz);
        set_ray(P, r, sx, sy, sz, tx, ty, tz);
        r.e = seed;
        r.stage = kStageSeed;
        return;
      }
    }
  }
  set_ray(P, r, x, y, z, tx, ty, tz);
  r.stage = kStageReloc;
}

// K1/K2/K3 of the reference folded into the prologue: pick the walk target.
PTB_HD void begin_particle(const WalkParams &P, int i, Ray &r, Counters &c, bool writer) {
  r.stage = kStageDone;
  const bool fly = P.flying ? (P.flying[i] == 1) : true;  // only the value 1 flies (Impl.cpp:95)
  if (!fly) return;  // dest := own origin => zero-length walk, nothing changes (Impl.cpp:100-102)
  const ParticleState s0 = load_state(P.state + i);
  const double x = s0.x, y = s0.y, z = s0.z;
  r.e = s0.elem;
  if (P.origin) {
    const double tx = PTB_LDG(P.origin + 3 * (size_t)i), ty = PTB_LDG(P.origin + 3 * (size_t)i + 1),
                 tz = PTB_LDG(P.origin + 3 * (size_t)i + 2);
    if (tx != x || ty != y || tz != z) {
      if (!all_finite(tx, ty, tz)) {  // unusable origin: the particle sits this move out
        if (writer) c.lost++;
        return;
      }
      start_reloc(P, r, x, y, z, tx, ty, tz);
      return;
    }
  }
  if (P.dest) start_tally(P, i, r, x, y, z, c, writer);
}

// The current ray ended (target reached, hull hit, or iteration limit).
// kReloadTarget: the caller does not keep Ray::tx,ty,tz alive in registers (the compact-layout
// kernel); the target is read back from the caller's array, where it came from: dest[] in the
// tally phase, origin[] in phase 1.  Same values, six registers fewer in the crossing loop.
template <bool kReloadTarget = false>
PTB_HD void end_ray(const WalkParams &P, int i, Ray &r, bool reached, double tnew, Counters &c,
                    bool writer) {
  // crossings of the ray that just ended: tally contributions in the tally phase, relocation crossings
  // otherwise (counted here, once per ray, instead of once per crossing)
  if (writer) {
    if (r.stage == kStageTally) c.segs += (unsigned)r.iters;
    else c.relocs += (unsigned)r.iters;
  }
  double x, y, z;
  if (kReloadTarget && (reached || r.stage == kStageSeed)) {
    const double *t = (r.stage == kStageTally ? P.dest : P.origin) + 3 * (size_t)i;
    r.tx = PTB_LDG(t); r.ty = PTB_LDG(t + 1); r.tz = PTB_LDG(t + 2);
  }
  if (r.stage == kStageSeed && !reached) {
    // the target is not reachable from the seed inside the mesh (it lies outside the hull):
    // redo phase 1 exactly as the reference does, from the particle's stored position
    const ParticleState s0 = load_state(P.state + i);
    x = s0.x; y = s0.y; z = s0.z;
    r.e = s0.elem;
    set_ray(P, r, x, y, z, r.tx, r.ty, r.tz);
    r.stage = kStageReloc;
    return;
  }
  if (reached) {  // tracer commit: origin <- dest, exactly (test lines 323-346)
    x = r.tx; y = r.ty; z = r.tz;
  } else {  // vacuum BC: dest <- intersection point (Impl.cpp:275-281)
    x = fma(tnew, r.ux, r.ox) + P.cx; y = fma(tnew, r.uy, r.oy) + P.cy; z = fma(tnew, r.uz, r.oz) + P.cz;
  }
  if (r.stage != kStageTally && P.dest) {
    start_tally(P, i, r, x, y, z, c, writer);  // phase 2 starts where phase 1 ended
  } else {
    if (writer) {
      store_state(P.state + i, x, y, z, r.e);
    }
    r.stage = kStageDone;
  }
}

// Functor body for one crossing, given the tracer's answer (texit, next).
template <bool kReloadTarget = false, bool kAggregateTally = false>
PTB_HD void advance(const WalkParams &P, int i, Ray &r, double texit, int32_t next, int32_t back,
                    Counters &c, bool writer) {
  const bool reached = !(texit < 1.0);  // last_exit == -1: destination inside this tet
  const double tnew = reached ? 1.0 : fmax(texit, r.tcur);
#if defined(__CUDA_ARCH__)
  if constexpr (kAggregateTally) {
    tally_add_aggregated(P.flux, r.e, (tnew - r.tcur) * r.wl, r.stage == kStageTally && writer);
  } else
#endif
  if (r.stage == kStageTally && writer)  // EvaluateFlux (Impl.cpp:362-379)
    PTB_TALLY_ADD(P.flux + r.e, (tnew - r.tcur) * r.wl);
  const bool hull = !reached && next < 0;  // next_elems == -1 (Impl.cpp:270-271)
  r.iters++;
  const bool over = r.iters >= P.max_iters;
  if (reached || hull || over) {
    if (over && !reached && !hull && writer && r.stage != kStageSeed) c.lost++;
    end_ray<kReloadTarget>(P, i, r, reached, tnew, c, writer);
  } else {
    r.e = next;  // UpdateCurrentElement (Impl.cpp:247-253)
    r.entry = back;
    r.tcur = tnew;
  }
}

}  // namespace ptb
