// Link-update kernels: one warp per record scores every entity of the record's block and draws the new link.
//
// Reference: updateEntityIdCollapsed GU:363-395 (PCG-II), updateEntityId / updateEntityIdSeq GU:399-466
// (PCG-I, Gibbs; dense form), DiscreteDist(weights).sample() GU:394,427,465.  Protocol: DESIGN.md section 4.
//
//   k_link_pcg2<A,NS> (dbl_link_pcg2.cuh) PCG-II, attributes fully unrolled (A = 1..16, NS non-constant): the block's entity table streams through
//                   shared memory in TE-entity tiles moved by TMA bulk copies (cp.async.bulk + mbarrier ring,
//                   one producer warp); per-record constants live in registers; the sparse similarity row of
//                   each record attribute is a perfect-hash table in shared memory (one bank-conflict-free
//                   probe per candidate and attribute).
//   k_link_match    PCG-I / Gibbs: same tile pipeline; candidates must agree on every observed non-distorted
//                   attribute, checked most-selective-first with a warp-wide early out.
//   k_link_generic  any A <= 32 / any row length; tiles read through L1/L2.  Fallback only.
#pragma once
#include <cuda_runtime.h>

#include <cstdint>

#include "dbl_internal.h"

constexpr int TE = 128;          // entities per tile of the block-sorted entity table
#ifndef DBL_LINK_WARPS
#define DBL_LINK_WARPS 8
#endif
constexpr int LINK_WARPS = DBL_LINK_WARPS;  // consumer warps (= records) per CTA
constexpr int MATCH_WARPS = 16;  // ... of k_link_match, which is bound by L2 -> shared-memory tile traffic
#ifndef DBL_LINK_STAGES
#define DBL_LINK_STAGES 4
#endif
constexpr int LINK_STAGES = DBL_LINK_STAGES;  // tile ring depth
constexpr int LINK_MAX_UNROLL_A = 16;
constexpr unsigned FULL = 0xffffffffu;

// int32 words per tile: A value rows (attribute-major), the f64 row N(e), one row of byte-packed constant attributes
__host__ __device__ inline size_t tile_words(int A) { return (size_t)A * TE + 3 * TE; }
// "Quad tiles" (k_link_pcg2): the words a lane needs about ONE candidate sit in groups of four, group-major
// ([group][slot][4] int32), so that a warp fetches a group with one conflict-free 128-bit load per lane.  Words of an
// entity: nv values (packed kernels: the NS non-constant values then the byte-packed constants; else all A values in
// kernel order) padded to a multiple of four; the f64 row N(e) follows the groups (8 contiguous bytes per lane: a
// 64-bit load of a word pair inside a 16-byte group would cost twice the wavefronts).
__host__ __device__ constexpr int qtile_nv(int A, int NS, bool packed) { return packed ? NS + 1 : A; }
__host__ __device__ constexpr int qtile_groups(int nv) { return (nv + 3) / 4; }
__host__ __device__ constexpr int qtile_words(int nv) { return qtile_groups(nv) * 4 + 2; }  // per entity

struct AttrDev {
  int V, is_const, kmax, hsize;
  int hshift, pad0, pad1, pad2;
  const double *phi, *probs, *norm, *invnorm, *pk, *cdf, *logphi, *lognorm, *expsim, *hvals;
  const double *diag;  // E(v, v) of every value (1 when the sparse row has no diagonal entry): no search per record
  const int *rowptr, *col, *hkeys;
  const unsigned *hmult;
};

// Control block of a context (device memory, 64-bit words): the sweep is enqueued without host round trips, so
// everything that changes from sweep to sweep is read from here by the kernels.
enum : int {
  CTL_ITER = 0,       // completed sweeps (= iteration of the state); the running sweep draws with CTL_ITER + 1
  CTL_STATUS = 1,     // 0 ok; bit 0 zero-mass categorical, bit 1 peer time-out, bit 2 a peer reported an error
  CTL_PAIRS = 2,      // (record, candidate) pairs visited by link kernels since context creation
  CTL_OWNED_ENT = 3,  // entities / records in the blocks this rank owns (prefix of ent_sorted / rec_sorted)
  CTL_OWNED_REC = 4,
  CTL_MOVED_ENT = 5,  // cluster messages sent in the last exchange
  CTL_MOVED_REC = 6,
  CTL_EPOCH = 7,      // barriers passed (peer-to-peer exchange)
  CTL_REPLACED = 8,   // block -> rank placements adopted by the device-side LPT
  CTL_WORK = 9,       // work counter of the persistent link kernel
  CTL_HEAVY = 10,     // records the pruned link kernel handed to k_link_heavy in the running sweep
  CTL_VALUES_REDO = 11,  // iteration of the last sweep in which k_values left a draw to k_values_log
  CTL_WORDS = 16
};
constexpr long long ST_ZERO_MASS = 1, ST_PEER_TIMEOUT = 2, ST_PEER_ERROR = 4;

struct LinkParams {
  int A, F, P, sampler;
  uint64_t seed;
  const long long *ctl;
  const AttrDev *attrs;
  const int *x, *file, *link;
  const unsigned *zmask;
  const double *theta;
  const int *ent_ptr, *tile_ptr, *rec_ptr, *cta_ptr, *ent_sorted, *rec_sorted;
  const int *tiles;
  const int *qtiles;         // quad tiles (k_link_pcg2)
  int qtile_pk;              // quad tiles hold the non-constant values + the byte-packed constants (else all A values)
  unsigned long long *work;  // k_link_pcg2: next group of records to take (persistent CTAs); zeroed before the launch
  double *lane_sums;         // k_link_pcg2: scratch, [CTA][consumer warp][32 chunks][32 lanes] pass-1 lane sums
  int *newlink;
  unsigned long long *status;  // &ctl[CTL_STATUS]
  unsigned long long *pairs;   // &ctl[CTL_PAIRS]
  // "kernel order" of the attributes: constant attributes first, then the others, each group in ascending
  // attribute id.  Tiles, per-record constants and the multiplication order of the protocol use this order.
  int perm[DBL_MAX_ATTRS];
  int pack_consts;         // tiles carry the byte-packed constant attributes (1..4 of them, vocabularies <= 255)
  const int *blk_of_link;  // block id of every entity (k_link_pruned: block of a record = block of its entity)
  int hslots, hshift;  // common size of the per-row similarity hash tables (k_link_pcg2); 0 = unavailable
};

// ---------------------------------------------------------------------------------------------------
// helpers
// ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ double shfl_xor_d(double v, int d) { return __shfl_xor_sync(FULL, v, d); }
__device__ __forceinline__ double shfl_up_d(double v, int d) { return __shfl_up_sync(FULL, v, d); }
__device__ __forceinline__ double shfl_d(double v, int l) { return __shfl_sync(FULL, v, l); }

// 5-level xor butterfly: every lane ends with the same sum
__device__ __forceinline__ double butterfly_sum(double v) {
  v = v + shfl_xor_d(v, 16);
  v = v + shfl_xor_d(v, 8);
  v = v + shfl_xor_d(v, 4);
  v = v + shfl_xor_d(v, 2);
  v = v + shfl_xor_d(v, 1);
  return v;
}

__device__ __forceinline__ bool row_find(const AttrDev &at, int v1, int v2, double &e) {
  int lo = at.rowptr[v1], hi = at.rowptr[v1 + 1] - 1;
  while (lo <= hi) {
    const int mid = (lo + hi) >> 1;
    const int c = at.col[mid];
    if (c == v2) { e = at.expsim[mid]; return true; }
    if (c < v2) lo = mid + 1; else hi = mid - 1;
  }
  return false;
}

__device__ __forceinline__ uint32_t link_iter(const LinkParams &p) { return (uint32_t)(p.ctl[CTL_ITER] + 1); }
// a failed sweep (zero-mass draw, peer error) is abandoned: every later kernel returns before it changes anything
__device__ __forceinline__ bool sweep_dead(const long long *ctl) { return ctl[CTL_STATUS] != 0; }

// CTA -> (block, first record) mapping shared by all link kernels
__device__ __forceinline__ int find_block(const LinkParams &p, int cta) {
  int lo = 0, hi = p.P;
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if (p.cta_ptr[mid] <= cta) lo = mid; else hi = mid;
  }
  return lo;
}

// Second half of the draw (DESIGN.md section 4.3): given the check-pointed running totals Q (lane c = end of
// chunk c) locate u*total: chunk -> lane (Kogge-Stone scan of the chunk's lane sums) -> step.  wf(j) must
// reproduce the pass-1 weight of candidate j bit for bit (0 for j >= n).
// lane_sums (optional): the lane sums of EVERY chunk as pass 1 produced them ([chunk][lane], this warp's scratch):
// the chosen chunk's sums are read back instead of being recomputed (1/nchunks of pass 1 per record otherwise).
template <class WeightFn>
__device__ __forceinline__ int finish_draw(int lane, int n, int nsteps, int spc, int nchunks, double Q, double total,
                                           double u, WeightFn wf, const double *lane_sums = nullptr) {
  const double t = u * total;
  unsigned m = __ballot_sync(FULL, lane < nchunks && Q > t);
  const int chunk = m ? (__ffs(m) - 1) : (nchunks - 1);
  double r = shfl_d(Q, chunk > 0 ? chunk - 1 : 0);
  if (chunk == 0) r = 0.0;
  const int s0 = chunk * spc, s1 = min(s0 + spc, nsteps);
  double ls = 0.0;
  if (lane_sums) ls = lane_sums[chunk * 32 + lane];
  else
    for (int s = s0; s < s1; ++s) ls = ls + wf((s << 5) + lane);
  double P = ls;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const double o = shfl_up_d(P, d);
    if (lane >= d) P = P + o;
  }
  m = __ballot_sync(FULL, r + P > t);
  int L;
  if (m) L = __ffs(m) - 1;
  else {
    const unsigned pos = __ballot_sync(FULL, ls > 0.0);
    L = pos ? (31 - __clz(pos)) : 0;
  }
  const double Pprev = shfl_up_d(P, 1);
  const double base_l = lane ? r + Pprev : r;
  const double base = shfl_d(base_l, L);
  double cum = 0.0;
  int step = -1, last_pos = -1;
  for (int g = s0; g < s1 && step < 0; g += 32) {
    const int s = g + lane;
    const double wi = (s < s1) ? wf((s << 5) + L) : 0.0;
    const int cnt = min(32, s1 - g);
    for (int i = 0; i < cnt; ++i) {
      const double wv = shfl_d(wi, i);
      cum = cum + wv;
      if (wv > 0.0) last_pos = g + i;
      if (base + cum > t) { step = g + i; break; }
    }
  }
  if (step < 0) step = last_pos >= 0 ? last_pos : s0;
  int j = (step << 5) + L;
  if (j >= n) j = n - 1;
  return j;
}

// ---------------------------------------------------------------------------------------------------
// generic kernel (fallback)
// ---------------------------------------------------------------------------------------------------
struct RecAttr {
  int kind;  // 0 skip, 1 const compare, 2 non-const sparse row, 3 missing non-const (PCG-II), 4 must match
  int x;
  int len;
  int pad;
  double rmatch;
  const int *col;
  const double *val;
  const double *tab;  // invnorm (kind 3) / norm (kind 2 of PCG-I)
};

// k = position in kernel order
__device__ __forceinline__ void prep_rec_attr(const LinkParams &p, int r, int k, RecAttr &c) {
  const int a = p.perm[k];
  const AttrDev &at = p.attrs[a];
  const int xv = p.x[(int64_t)r * p.A + a];
  c.kind = 0; c.x = xv; c.len = 0; c.pad = 0; c.rmatch = 1.0; c.col = nullptr; c.val = nullptr; c.tab = nullptr;
  if (p.sampler == DBL_PCG_II) {
    if (xv < 0) {
      if (!at.is_const) { c.kind = 3; c.tab = at.invnorm; }
    } else {
      const double th = p.theta[a * p.F + p.file[r]];
      double d = th * at.phi[xv];
      if (at.is_const) {
        c.kind = 1;
        c.rmatch = 1.0 + (1.0 - th) / d;
        c.rmatch = (c.rmatch - 1.0) + 1.0;  // see k_link_pcg2: the multiplier is rebuilt from (rmatch - 1)
      } else {
        d = d * at.norm[xv];
        const double ediag = at.diag[xv];
        c.kind = 2;
        c.rmatch = ediag + (1.0 - th) / d;
        c.rmatch = (c.rmatch - 1.0) + 1.0;
        c.col = at.col + at.rowptr[xv];
        c.val = at.expsim + at.rowptr[xv];
        c.len = at.rowptr[xv + 1] - at.rowptr[xv];
      }
    }
  } else if (xv >= 0) {
    const bool dist = (p.zmask[r] >> a) & 1u;
    if (!dist) c.kind = 4;
    else if (!at.is_const) {
      c.kind = 2;
      c.tab = at.norm;
      c.col = at.col + at.rowptr[xv];
      c.val = at.expsim + at.rowptr[xv];
      c.len = at.rowptr[xv + 1] - at.rowptr[xv];
    }
  }
}

__device__ __forceinline__ bool rec_row_find(const RecAttr &c, int yv, double &e) {
  int lo = 0, hi = c.len - 1;
  while (lo <= hi) {
    const int mid = (lo + hi) >> 1;
    const int cv = c.col[mid];
    if (cv == yv) { e = c.val[mid]; return true; }
    if (cv < yv) lo = mid + 1; else hi = mid - 1;
  }
  return false;
}

// protocol weight of one candidate; ycol points at attribute 0 of the candidate inside its tile (stride TE)
__device__ __forceinline__ double generic_weight(const RecAttr *ra, int A, bool pcg2, const int *ycol, double N) {
  double w;
  if (pcg2) {
    double c = 1.0;  // the constant attributes form their own product (a table look-up in k_link_pcg2)
    for (int a = 0; a < A; ++a)
      if (ra[a].kind == 1 && ycol[a * TE] == ra[a].x) c = c * ra[a].rmatch;
    w = N * c;
    for (int a = 0; a < A; ++a) {  // non-constant attributes: one factor each, equal (multiplier) or similar (exp sim)
      if (ra[a].kind != 2) continue;
      const int yv = ycol[a * TE];
      double e;
      if (yv == ra[a].x) w = w * ra[a].rmatch;
      else if (rec_row_find(ra[a], yv, e)) w = w * e;
    }
    for (int a = 0; a < A; ++a)
      if (ra[a].kind == 3) w = w * ra[a].tab[ycol[a * TE]];
  } else {
    for (int a = 0; a < A; ++a)
      if (ra[a].kind == 4 && ycol[a * TE] != ra[a].x) return 0.0;
    w = 1.0;
    for (int a = 0; a < A; ++a)
      if (ra[a].kind == 2) w = w * ra[a].tab[ycol[a * TE]];
    for (int a = 0; a < A; ++a) {
      double e;
      if (ra[a].kind == 2 && rec_row_find(ra[a], ycol[a * TE], e)) w = w * e;
    }
  }
  return w;
}

// visited = (record, candidate) pairs this record looked at: the block's entity count in the dense kernels, the
// length of the posting list walked in the pruned one
__device__ __forceinline__ void store_link(const LinkParams &p, int lane, int r, int b, long long visited, int j) {
  if (lane == 0) {
    p.newlink[r] = p.ent_sorted[p.ent_ptr[b] + j];
    atomicAdd(p.pairs, (unsigned long long)visited);
  }
}
__device__ __forceinline__ void fail_link(const LinkParams &p, int lane, int r) {
  if (lane == 0) {  // reference: IllegalArgumentException("zero probability mass")
    atomicOr(p.status, (unsigned long long)ST_ZERO_MASS);
    p.newlink[r] = p.link[r];
  }
}

#ifdef DBL_ENGINE_TU  // non-template kernels live in exactly one translation unit (dbl_engine.cu)
__global__ void __launch_bounds__(LINK_WARPS * 32) k_link_generic(LinkParams p) {
  __shared__ RecAttr s_ra[LINK_WARPS][DBL_MAX_ATTRS];
  const int cta = blockIdx.x;
  if (sweep_dead(p.ctl) || cta >= p.cta_ptr[p.P]) return;
  const int b = find_block(p, cta);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int ridx = p.rec_ptr[b] + (cta - p.cta_ptr[b]) * LINK_WARPS + warp;
  if (ridx >= p.rec_ptr[b + 1]) return;
  const int r = p.rec_sorted[ridx];
  const int A = p.A;
  const bool pcg2 = (p.sampler == DBL_PCG_II);
  RecAttr *ra = s_ra[warp];
  if (lane < A) {
    RecAttr c;
    prep_rec_attr(p, r, lane, c);
    ra[lane] = c;
  }
  __syncwarp();
  const int n = p.ent_ptr[b + 1] - p.ent_ptr[b];
  const int ntiles = (n + TE - 1) / TE;
  const int nsteps = ntiles * (TE / 32);                       // steps beyond the last candidate add zeros
  const int spc = (TE / 32) * max(1, (ntiles + 31) >> 5);      // a chunk is a whole number of tiles
  const int nchunks = (nsteps + spc - 1) / spc;
  const size_t tw = tile_words(A);
  const int *tiles = p.tiles + (size_t)p.tile_ptr[b] * tw;
  auto wf = [&](int j) -> double {
    if (j >= n) return 0.0;
    const int *tile = tiles + (size_t)(j / TE) * tw;
    const int slot = j % TE;
    const double N = reinterpret_cast<const double *>(tile + (size_t)A * TE)[slot];
    return generic_weight(ra, A, pcg2, tile + slot, N);
  };
  double run = 0.0, Q = 0.0, acc = 0.0;
  int mark = min(spc, nsteps), chunk = 0;
  for (int s = 0; s < nsteps; ++s) {
    acc = acc + wf((s << 5) + lane);
    if (s + 1 == mark) {
      run = run + butterfly_sum(acc);
      if (lane == chunk) Q = run;
      ++chunk;
      acc = 0.0;
      mark = min(mark + spc, nsteps);
    }
  }
  if (!(run > 0.0) || isinf(run)) { fail_link(p, lane, r); return; }
  const U2 u = uniform2(p.seed, PH_LINK, link_iter(p), (uint32_t)r, 0u);
  const int j = finish_draw(lane, n, nsteps, spc, nchunks, Q, run, u.u0, wf);
  store_link(p, lane, r, b, n, j);
}

#endif  // DBL_ENGINE_TU

// ---------------------------------------------------------------------------------------------------
// TMA / mbarrier plumbing (sm_90+ PTX; SASS: UBLKCP, SYNCS)
// ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t *bar, unsigned count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t *bar, unsigned bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// consumer-side wait (critical path): plain try_wait loop -- the hardware suspends the warp for a short,
// implementation-defined time per attempt and wakes it promptly when the phase completes
__device__ __forceinline__ void mbar_wait(uint64_t *bar, unsigned parity) {
  const uint32_t addr = smem_u32(bar);
  uint32_t ok = 0;
  while (!ok) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(addr), "r"(parity)
        : "memory");
  }
}
#ifndef DBL_PRODUCER_HINT
#define DBL_PRODUCER_HINT 0x989680u
#endif
// producer-side wait (off the critical path while the ring is full): long suspend-time hint so that the idle
// producer lane does not steal issue slots from the consumer warps
__device__ __forceinline__ void mbar_wait_relaxed(uint64_t *bar, unsigned parity) {
  const uint32_t addr = smem_u32(bar);
  uint32_t ok = 0;
  while (!ok) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\tselp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(addr), "r"(parity), "r"(DBL_PRODUCER_HINT)
        : "memory");
  }
}
__device__ __forceinline__ void tma_load_1d(void *smem_dst, const void *gsrc, unsigned bytes, uint64_t *bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(smem_dst)),
               "l"(gsrc), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

// Shared-memory ring of entity tiles filled by one producer warp; every consumer warp of the CTA reads every tile.
struct TileRing {
  int *tiles;          // LINK_STAGES * tile_words
  uint64_t *full;      // LINK_STAGES
  uint64_t *empty;     // LINK_STAGES
  int tw;              // words per tile
};

__device__ __forceinline__ void ring_init(const TileRing &rg, int consumers, int producers = 1) {
  if (threadIdx.x == 0) {
    for (int s = 0; s < LINK_STAGES; ++s) { mbar_init(&rg.full[s], producers); mbar_init(&rg.empty[s], consumers); }
    mbar_fence_init();
  }
  __syncthreads();
}
// producer: one lane streams ntiles tiles from global
// RELAXED: the consumers are slow (PCG-II): let the producer sleep.  !RELAXED: the consumers drain tiles faster
// than the producer can be woken (PCG-I): poll.
// base = tiles this CTA has already streamed through the ring (persistent CTAs): stages and phases continue
template <bool RELAXED>
__device__ __forceinline__ void ring_produce(const TileRing &rg, const int *gsrc, int ntiles, int base = 0) {
  const unsigned bytes = (unsigned)rg.tw * 4u;
  for (int t = 0; t < ntiles; ++t) {
    const int g = base + t;
    const int s = g % LINK_STAGES;
    if (g >= LINK_STAGES) {
      if (RELAXED) mbar_wait_relaxed(&rg.empty[s], ((g / LINK_STAGES) - 1) & 1);
      else mbar_wait(&rg.empty[s], ((g / LINK_STAGES) - 1) & 1);
    }
    mbar_arrive_expect_tx(&rg.full[s], bytes);
    tma_load_1d(rg.tiles + (size_t)s * rg.tw, gsrc + (size_t)t * rg.tw, bytes, &rg.full[s]);
  }
}

// The same ring filled with 16-byte cp.async copies by all 32 lanes of the producer warp (SASS LDGSTS) instead of one
// bulk copy per tile: every lane's copies arrive on the stage's barrier (initialised with 32 producers).
__device__ __forceinline__ void ring_produce_ldgsts(const TileRing &rg, const int *gsrc, int ntiles, int base, int lane) {
  const int vecs = rg.tw / 4;  // 16-byte pieces per tile
  for (int t = 0; t < ntiles; ++t) {
    const int g = base + t;
    const int s = g % LINK_STAGES;
    if (g >= LINK_STAGES) mbar_wait_relaxed(&rg.empty[s], ((g / LINK_STAGES) - 1) & 1);
    const int *src = gsrc + (size_t)t * rg.tw;
    int *dst = rg.tiles + (size_t)s * rg.tw;
    for (int i = lane; i < vecs; i += 32)
      asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(dst + i * 4)), "l"(src + i * 4) : "memory");
    asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(smem_u32(&rg.full[s])) : "memory");
  }
}

// ---------------------------------------------------------------------------------------------------
// k_link_match: PCG-I / Gibbs (GU:399-466).  A candidate has weight 0 unless it agrees with the record on every
// observed, non-distorted attribute; the agreeing few are scored with the generic weight function.
// ---------------------------------------------------------------------------------------------------
#ifdef DBL_ENGINE_TU
__global__ void __launch_bounds__((MATCH_WARPS + 1) * 32) k_link_match(LinkParams p) {
  extern __shared__ __align__(128) unsigned char smem[];
  __shared__ RecAttr s_ra[MATCH_WARPS][DBL_MAX_ATTRS];
  __shared__ int s_mm_attr[MATCH_WARPS][DBL_MAX_ATTRS];  // must-match attributes, most selective first
  __shared__ int s_mm_x[MATCH_WARPS][DBL_MAX_ATTRS];
  const int cta = blockIdx.x;
  if (sweep_dead(p.ctl) || cta >= p.cta_ptr[p.P]) return;
  const int b = find_block(p, cta);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int A = p.A;
  const int n = p.ent_ptr[b + 1] - p.ent_ptr[b];
  const int ntiles = p.tile_ptr[b + 1] - p.tile_ptr[b];
  const int TW = (int)tile_words(A);
  TileRing rg;
  rg.tiles = reinterpret_cast<int *>(smem);
  rg.full = reinterpret_cast<uint64_t *>(smem + (size_t)LINK_STAGES * TW * 4);
  rg.empty = rg.full + LINK_STAGES;
  rg.tw = TW;
  const int *gtiles = p.tiles + (size_t)p.tile_ptr[b] * TW;
  ring_init(rg, MATCH_WARPS);
  if (warp == MATCH_WARPS) {
    if (lane == 0) ring_produce<false>(rg, gtiles, ntiles);
    return;
  }
  const int ridx = p.rec_ptr[b] + (cta - p.cta_ptr[b]) * MATCH_WARPS + warp;
  const bool active = ridx < p.rec_ptr[b + 1];
  const int r = active ? p.rec_sorted[ridx] : -1;
  RecAttr *ra = s_ra[warp];
  int nmm = 0;
  if (active) {
    double sel = 2.0;  // selectivity key: phi(x) of a must-match attribute
    bool mm = false;
    if (lane < A) {
      RecAttr c;
      prep_rec_attr(p, r, lane, c);
      ra[lane] = c;
      mm = (c.kind == 4);
      if (mm) sel = p.attrs[p.perm[lane]].phi[c.x];
    }
    // rank must-match attributes by (phi, attribute id): tiny all-pairs rank via shuffles
    int rank = 0;
    for (int o = 0; o < A; ++o) {
      const double so = shfl_d(sel, o);
      const bool mo = __shfl_sync(FULL, (int)mm, o);
      if (mo && (so < sel || (so == sel && o < lane))) ++rank;
    }
    if (mm) { s_mm_attr[warp][rank] = lane; s_mm_x[warp][rank] = ra[lane].x; }
    nmm = __popc(__ballot_sync(FULL, mm));
    __syncwarp();
  }
  const int nsteps = ntiles * (TE / 32);
  const int tpc = max(1, (ntiles + 31) >> 5);
  const int spc = (TE / 32) * tpc;
  const int nchunks = (nsteps + spc - 1) / spc;
  const int *mma = s_mm_attr[warp];
  const int *mmx = s_mm_x[warp];
  const int off0 = nmm ? mma[0] * TE : 0;
  const int x0 = nmm ? mmx[0] : 0;

  double run = 0.0, Q = 0.0, acc = 0.0;
  int chunk = 0, tile_in_chunk = 0;
  for (int t = 0; t < ntiles; ++t) {
    const int s = t % LINK_STAGES;
    mbar_wait(&rg.full[s], (t / LINK_STAGES) & 1);
    if (active) {
      const int *tile = rg.tiles + (size_t)s * TW;
      const double *tileN = reinterpret_cast<const double *>(tile + A * TE);
      const int valid = min(TE, n - t * TE);  // candidates in this tile (the last tile is zero padded)
#pragma unroll
      for (int q = 0; q < TE / 32; ++q) {
        const int slot = q * 32 + lane;
        // the most selective must-match attribute decides almost every candidate: one load, one compare, one vote
        bool ok = (slot < valid) && (nmm == 0 || tile[off0 + slot] == x0);
        if (__any_sync(FULL, ok)) {
          for (int k = 1; k < nmm; ++k) {
            ok = ok && (tile[mma[k] * TE + slot] == mmx[k]);
            if (!__any_sync(FULL, ok)) break;  // warp-uniform: nobody left after this attribute
          }
          if (ok) acc = acc + generic_weight(ra, A, false, tile + slot, tileN[slot]);
        }
      }
      if (++tile_in_chunk == tpc || t + 1 == ntiles) {
        run = run + butterfly_sum(acc);
        if (lane == chunk) Q = run;
        ++chunk;
        acc = 0.0;
        tile_in_chunk = 0;
      }
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(&rg.empty[s]);
  }
  if (!active) return;
  if (!(run > 0.0) || isinf(run)) { fail_link(p, lane, r); return; }
  auto wf = [&](int j) -> double {
    if (j >= n) return 0.0;
    const int *tile = gtiles + (size_t)(j / TE) * TW;
    const int slot = j % TE;
    return generic_weight(ra, A, false, tile + slot, reinterpret_cast<const double *>(tile + (size_t)A * TE)[slot]);
  };
  const U2 u = uniform2(p.seed, PH_LINK, link_iter(p), (uint32_t)r, 0u);
  const int j = finish_draw(lane, n, nsteps, spc, nchunks, Q, run, u.u0, wf);
  store_link(p, lane, r, b, n, j);
}
#endif  // DBL_ENGINE_TU

// ---------------------------------------------------------------------------------------------------
// k_link_pruned: PCG-I / Gibbs with a per-sweep inverted index (the reference prunes the same way:
// EntityInvertedIndex GU:41-76, getPossibleEntities GU:473-530 -- smallest posting list first).  Only the
// candidates that agree with the record on its most selective observed non-distorted attribute are visited;
// every other candidate has weight exactly 0 in the dense kernel, and adding +0.0 never changes a sum, so the
// lane sums, chunk totals and the draw are bit-identical to k_link_match / k_link_generic.
// Index: entries (key = (block*A + kernel attribute) << 32 | value, payload = candidate position j) sorted by
// key, positions ascending inside a key.
// ---------------------------------------------------------------------------------------------------
#ifdef DBL_ENGINE_TU
// key = ((block * A + kernel attribute) << vbits) | value; rows this rank does not own go to the dummy block P
__global__ void k_inv_keys(int64_t E, int A, int P, int vbits, const int *__restrict__ y,
                           const int *__restrict__ blk_sorted, const int *__restrict__ ent_sorted,
                           const int *__restrict__ ent_ptr, const int *__restrict__ perm,
                           unsigned long long *__restrict__ key, int *__restrict__ pos) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= E * A) return;
  const int64_t i = t / A;
  const int k = (int)(t % A);
  const int b = min(blk_sorted[i], P);
  const int e = ent_sorted[i];
  const unsigned long long v = (b < P) ? (unsigned)y[(int64_t)e * A + perm[k]] : 0u;
  key[t] = ((unsigned long long)((unsigned)b * (unsigned)A + (unsigned)k) << vbits) | v;
  pos[t] = (b < P) ? (int)(i - ent_ptr[b]) : -1;
}

// seg[g] = first index entry of group g = block * A + kernel attribute (one pass over the sorted keys)
__global__ void k_inv_segments(int64_t n, int n_groups, int vbits, const unsigned long long *__restrict__ key,
                               int *__restrict__ seg) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i > n) return;
  const int cur = (i < n) ? (int)min((unsigned long long)n_groups, key[i] >> vbits) : n_groups;
  const int prev = (i > 0) ? (int)min((unsigned long long)n_groups, key[i - 1] >> vbits) : -1;
  for (int g = prev + 1; g <= cur; ++g) seg[g] = (int)i;
}

// vptr[(block * sumV) + voff[kernel attribute] + value] = first index entry of that (block, attribute, value); the
// table is dense (values without entities get an empty range), so a record finds a posting list with two loads
struct InvDense {
  int A, sumV, vbits;
  int voff[DBL_MAX_ATTRS];
};

// The same index with 32-bit keys = the dense (block, attribute, value) id itself, over ALL E * A slots of the sorted
// entity table: rows of blocks this rank does not own get ids beyond n_ids and sort to the end.  Nothing here
// depends on how many entities the rank owns, so a sharded sweep needs no read-back to size the sort.  The ids
// beyond n_ids are spread over the rest of the key range (`spread` values): with ONE sentinel value 7/8 of the keys of an 8-rank shard were
// equal, and a radix sort whose items all fall into one bin serialises on that bin (PCG-I went from 430 sweeps/s on
// 4 GPUs to 280 on 8).
__global__ void k_inv_keys32(int64_t E, int A, int P, InvDense d, long long n_ids, long long spread, const int *__restrict__ y,
                             const int *__restrict__ blk_sorted, const int *__restrict__ ent_sorted,
                             const int *__restrict__ ent_ptr, const int *__restrict__ perm,
                             unsigned *__restrict__ key, int *__restrict__ pos) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= E * A) return;
  const int64_t i = t / A;
  const int k = (int)(t % A);
  const int b = blk_sorted[i];
  if (b < P) {
    const int e = ent_sorted[i];
    key[t] = (unsigned)((long long)b * d.sumV + d.voff[k] + y[(int64_t)e * A + perm[k]]);
    pos[t] = (int)(i - ent_ptr[b]);
  } else {
    key[t] = (unsigned)(n_ids + t % spread);
    pos[t] = -1;
  }
}
// vptr[id] = first sorted entry whose key is >= id.  The thread at a boundary between two different keys fills the ids
// in between.  On a shard the keys of whole blocks are missing (7/8 of the id space on 8 ranks): a boundary thread
// filled up to ~2 million entries one after the other, and the sharded PCG-I sweep got SLOWER with every rank added
// (link phase 1.2 ms on 2 GPUs, 1.4-1.7 ms on 4).  Nothing ever looks up an id of a block without entities (a record
// queries ids of its own block b, and id + 1 <= (b + 1) * sumV), so the gap is filled only to the first id of the
// block after the previous key's and from the first id of the current key's block.
__global__ void k_inv_value_ptr32(int64_t n, long long n_ids, long long sumV, const unsigned *__restrict__ key,
                                  int *__restrict__ vptr) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i > n) return;
  const long long cur = (i < n) ? min((long long)key[i], n_ids) : n_ids;
  const long long prev = (i > 0) ? min((long long)key[i - 1], n_ids) : -1;
  if (cur == prev) return;
  const long long pb = prev >= 0 ? prev / sumV : -1, cb = cur / sumV;
  if (cb > pb + 1) {
    const long long e1 = min((pb + 1) * sumV, cur);
    for (long long g = prev + 1; g <= e1; ++g) vptr[g] = (int)i;
    for (long long g = max(cb * sumV, e1 + 1); g <= cur; ++g) vptr[g] = (int)i;
  } else {
    for (long long g = prev + 1; g <= cur; ++g) vptr[g] = (int)i;
  }
}

__device__ __forceinline__ int64_t inv_lower_bound(const unsigned long long *__restrict__ key, int64_t lo, int64_t hi,
                                                   unsigned long long want) {
  while (lo < hi) {
    const int64_t mid = (lo + hi) >> 1;
    if (key[mid] < want) lo = mid + 1; else hi = mid;
  }
  return lo;
}

struct PrunedParams {
  LinkParams lp;
  const unsigned long long *inv_key;
  const int *inv_pos;
  long long inv_n;
  long long R;
  int vbits;
  const int *rec_key_sorted;  // block-major sort key of rec_sorted[i]
  int rec_key_shift;
  const int *inv_vptr;  // dense (block, attribute, value) -> first entry; nullptr: binary search inside inv_seg
  int sumV;
  int voff[DBL_MAX_ATTRS];
  const int *inv_seg;  // (P+1)*A + 1 group offsets
  int *heavy_list;     // positions (in rec_sorted) of the records left to k_link_heavy; count in ctl[CTL_HEAVY]
};

// A record without any must-match attribute (every observed attribute distorted) has to score its whole block.  One
// warp doing that is the tail of the whole kernel (RLdata10000 in steady state: one such record in a 2 500-entity
// block = 0.75 ms against 25 us for everything else), so blocks beyond this size leave those records to k_link_heavy,
// a CTA per record.
constexpr int HEAVY_MIN_CANDIDATES = 256;
constexpr int HEAVY_WARPS = 16;

constexpr int PRUNED_SCAP = 48;  // survivors kept for pass 2 (more than that: pass 2 walks the postings again)
struct PrunedShared {
  RecAttr ra[LINK_WARPS][DBL_MAX_ATTRS];
  int mm_attr[LINK_WARPS][DBL_MAX_ATTRS];
  int mm_x[LINK_WARPS][DBL_MAX_ATTRS];
  int sj[LINK_WARPS][PRUNED_SCAP];
  double sw[LINK_WARPS][PRUNED_SCAP];
};

// one record (position ridx of rec_sorted) by one warp
__device__ __forceinline__ void pruned_record(const PrunedParams &pp, PrunedShared &sh, long long ridx, int warp, int lane) {
  constexpr int SCAP = PRUNED_SCAP;
  RecAttr (&s_ra)[LINK_WARPS][DBL_MAX_ATTRS] = sh.ra;
  int (&s_mm_attr)[LINK_WARPS][DBL_MAX_ATTRS] = sh.mm_attr;
  int (&s_mm_x)[LINK_WARPS][DBL_MAX_ATTRS] = sh.mm_x;
  int (&s_sj)[LINK_WARPS][SCAP] = sh.sj;
  double (&s_sw)[LINK_WARPS][SCAP] = sh.sw;
  const LinkParams &p = pp.lp;
  const int r = p.rec_sorted[ridx];
  const int b = pp.rec_key_sorted[ridx] >> pp.rec_key_shift;  // the sort key of the record: block id above the cost class
  const int A = p.A;
  const int n = p.ent_ptr[b + 1] - p.ent_ptr[b];
  const int ntiles = p.tile_ptr[b + 1] - p.tile_ptr[b];
  const size_t TW = tile_words(A);
  const int *gtiles = p.tiles + (size_t)p.tile_ptr[b] * TW;
  RecAttr *ra = s_ra[warp];
  int nmm = 0;
  bool has_sim = false;  // some observed distorted non-constant attribute: weights are not all 1
  long long plo = 0, phi = n;  // posting range in the index, or the whole block when nothing must match
  int best = -1;
  {
    bool mm = false;
    long long lo = 0, len = 0x7fffffffffffLL;
    if (lane < A) {
      RecAttr c;
      prep_rec_attr(p, r, lane, c);
      ra[lane] = c;
      mm = (c.kind == 4);
      if (mm) {
        if (pp.inv_vptr) {
          const long long id = (long long)b * pp.sumV + pp.voff[lane] + c.x;
          lo = pp.inv_vptr[id];
          len = pp.inv_vptr[id + 1] - lo;
        } else {
          const unsigned long long base = (unsigned long long)((unsigned)b * (unsigned)A + (unsigned)lane) << pp.vbits;
          const int g = b * A + lane;
          const long long s0 = pp.inv_seg[g], s1 = pp.inv_seg[g + 1];  // the E_b entries of (block, attribute)
          lo = inv_lower_bound(pp.inv_key, s0, s1, base | (unsigned)c.x);
          const long long hi = inv_lower_bound(pp.inv_key, lo, s1, base | ((unsigned)c.x + 1u));
          len = hi - lo;
        }
      }
    }
    const unsigned mmask = __ballot_sync(FULL, mm);
    nmm = __popc(mmask);
    has_sim = __any_sync(FULL, lane < A && ra[lane].kind == 2);
    if (mm) {
      const int rank = __popc(mmask & ((1u << lane) - 1u));
      s_mm_attr[warp][rank] = lane;
      s_mm_x[warp][rank] = ra[lane].x;
    }
    // shortest posting list (ties: lowest attribute)
    long long bl = len;
    int bk = mm ? lane : 64;
#pragma unroll
    for (int d = 16; d >= 1; d >>= 1) {
      const long long ol = __shfl_xor_sync(FULL, bl, d);
      const int ok = __shfl_xor_sync(FULL, bk, d);
      if (ol < bl || (ol == bl && ok < bk)) { bl = ol; bk = ok; }
    }
    if (nmm > 0) {
      best = bk;
      plo = __shfl_sync(FULL, lo, best);
      phi = plo + bl;
    }
    __syncwarp();
  }
  if (nmm == 0 && n > HEAVY_MIN_CANDIDATES) {
    if (lane == 0) pp.heavy_list[atomicAdd(reinterpret_cast<unsigned long long *>(const_cast<long long *>(p.ctl) + CTL_HEAVY), 1ull)] = (int)ridx;
    return;
  }
  const int *mma = s_mm_attr[warp];
  const int *mmx = s_mm_x[warp];
  const int nsteps = ntiles * (TE / 32);
  const int tpc = max(1, (ntiles + 31) >> 5);
  const int spc = (TE / 32) * tpc;
  const int nchunks = (nsteps + spc - 1) / spc;
  const int cand_per_chunk = TE * tpc;

  // candidate j of index entry idx, its protocol weight (0 unless it survives every must-match attribute)
  auto cand_weight = [&](long long idx, int &j) -> double {
    j = -1;
    if (idx >= phi) return 0.0;
    j = (nmm > 0) ? pp.inv_pos[idx] : (int)idx;
    const int *tile = gtiles + (size_t)(j / TE) * TW;
    const int slot = j % TE;
    bool ok = true;
    for (int k = 0; k < nmm && ok; ++k)
      if (mma[k] != best) ok = (tile[mma[k] * TE + slot] == mmx[k]);
    if (!ok) return 0.0;
    if (!has_sim) return 1.0;  // GU:408-411: uniform over the candidates
    return generic_weight(ra, A, false, tile + slot, reinterpret_cast<const double *>(tile + (size_t)A * TE)[slot]);
  };

  // ---- pass 1: lane sums per chunk from the survivors only
  double run = 0.0, Q = 0.0, s = 0.0;
  int cur = 0;
  bool dirty = false;
  auto close_chunks_until = [&](int c_next) {  // finalise chunks cur .. c_next-1 (only `cur` can hold mass)
    if (cur < c_next) {
      if (dirty) { run = run + butterfly_sum(s); s = 0.0; dirty = false; }
      if (lane >= cur && lane < c_next) Q = run;
      cur = c_next;
    }
  };
  int ns = 0;  // survivors seen (stored while they fit)
  auto add_survivor = [&](int ji, double wi) {
    close_chunks_until(ji / cand_per_chunk);
    if (lane == (ji & 31)) s = s + wi;
    dirty = true;
    if (ns < SCAP && lane == 0) { s_sj[warp][ns] = ji; s_sw[warp][ns] = wi; }
    ++ns;
  };
  if (nmm > 1) {
    // every lane tests its posting against ONE other must-match attribute; the few that pass are then checked
    // by the whole warp, one attribute per lane, so a survivor costs one more load instead of a chain of them
    int k1 = (mma[0] != best) ? 0 : 1;
    const int a1 = mma[k1], x1 = mmx[k1];
    for (long long g = plo; g < phi; g += 32) {
      const long long idx = g + lane;
      int j = -1;
      bool pass = false;
      if (idx < phi) {
        j = pp.inv_pos[idx];
        pass = (gtiles[(size_t)(j / TE) * TW + a1 * TE + (j % TE)] == x1);
      }
      unsigned live = __ballot_sync(FULL, pass);
      while (live) {
        const int i = __ffs(live) - 1;
        live &= live - 1;
        const int ji = __shfl_sync(FULL, j, i);
        const int *tile = gtiles + (size_t)(ji / TE) * TW;
        const int slot = ji % TE;
        bool okl = true;
        if (lane < nmm && mma[lane] != best) okl = (tile[mma[lane] * TE + slot] == mmx[lane]);
        if (!__all_sync(FULL, okl)) continue;
        const double wi = has_sim ? generic_weight(ra, A, false, tile + slot,
                                                   reinterpret_cast<const double *>(tile + (size_t)A * TE)[slot])
                                  : 1.0;  // GU:408-411: uniform over the candidates
        if (wi > 0.0) add_survivor(ji, wi);
      }
    }
  } else {
    for (long long g = plo; g < phi; g += 32) {
      int j;
      const double w = cand_weight(g + lane, j);
      unsigned live = __ballot_sync(FULL, w > 0.0);
      while (live) {
        const int i = __ffs(live) - 1;
        live &= live - 1;
        add_survivor(__shfl_sync(FULL, j, i), shfl_d(w, i));
      }
    }
  }
  __syncwarp();
  if (ns == 1) {  // a single candidate with positive weight is drawn whatever the uniform is: skip the search
    if (isinf(s_sw[warp][0])) { fail_link(p, lane, r); return; }
    store_link(p, lane, r, b, phi - plo, s_sj[warp][0]);
    return;
  }
  close_chunks_until(nchunks);
  if (!(run > 0.0) || isinf(run)) { fail_link(p, lane, r); return; }

  // ---- pass 2: the same walk restricted to the chosen chunk
  const U2 u = uniform2(p.seed, PH_LINK, link_iter(p), (uint32_t)r, 0u);
  const double t = u.u0 * run;
  unsigned m = __ballot_sync(FULL, lane < nchunks && Q > t);
  const int chunk = m ? (__ffs(m) - 1) : (nchunks - 1);
  double rsum = shfl_d(Q, chunk > 0 ? chunk - 1 : 0);
  if (chunk == 0) rsum = 0.0;
  const bool stored = (ns <= SCAP);
  double ls = 0.0;
  if (stored) {
    for (int i = 0; i < ns; ++i) {
      const int ji = s_sj[warp][i];
      if (ji / cand_per_chunk == chunk && lane == (ji & 31)) ls = ls + s_sw[warp][i];
    }
  } else {
    for (long long g = plo; g < phi; g += 32) {
      int j;
      const double w = cand_weight(g + lane, j);
      unsigned live = __ballot_sync(FULL, w > 0.0 && j / cand_per_chunk == chunk);
      while (live) {
        const int i = __ffs(live) - 1;
        live &= live - 1;
        const int ji = __shfl_sync(FULL, j, i);
        const double wi = shfl_d(w, i);
        if (lane == (ji & 31)) ls = ls + wi;
      }
    }
  }
  double Pfx = ls;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const double o = shfl_up_d(Pfx, d);
    if (lane >= d) Pfx = Pfx + o;
  }
  m = __ballot_sync(FULL, rsum + Pfx > t);
  int L;
  if (m) L = __ffs(m) - 1;
  else {
    const unsigned pos = __ballot_sync(FULL, ls > 0.0);
    L = pos ? (31 - __clz(pos)) : 0;
  }
  const double Pprev = shfl_up_d(Pfx, 1);
  const double base_l = lane ? rsum + Pprev : rsum;
  const double base = shfl_d(base_l, L);
  double cum = 0.0;
  int pick = -1, last_pos = -1;
  if (stored) {
    for (int i = 0; i < ns && pick < 0; ++i) {
      const int ji = s_sj[warp][i];
      if (ji / cand_per_chunk == chunk && (ji & 31) == L) {
        cum = cum + s_sw[warp][i];
        last_pos = ji;
        if (base + cum > t) pick = ji;
      }
    }
  } else {
    for (long long g = plo; g < phi && pick < 0; g += 32) {
      int j;
      const double w = cand_weight(g + lane, j);
      unsigned live = __ballot_sync(FULL, w > 0.0 && j / cand_per_chunk == chunk && (j & 31) == L);
      while (live) {
        const int i = __ffs(live) - 1;
        live &= live - 1;
        const int ji = __shfl_sync(FULL, j, i);
        const double wi = shfl_d(w, i);
        cum = cum + wi;
        last_pos = ji;
        if (base + cum > t) { pick = ji; break; }
      }
    }
  }
  if (pick < 0) pick = last_pos >= 0 ? last_pos : (chunk * cand_per_chunk + L < n ? chunk * cand_per_chunk + L : n - 1);
  store_link(p, lane, r, b, phi - plo, pick);
}

// A fixed grid of warps strides over the records of the blocks this rank owns (they come first in rec_sorted; the
// count is read on the device).  One CTA per 8 records of the WHOLE data set, most of them returning at once on a
// shard, cost more than it looks: 0.2 ms of a 0.9 ms kernel on 2 GPUs, and growing with the rank count.
__global__ void __launch_bounds__(LINK_WARPS * 32) k_link_pruned(PrunedParams pp) {
  __shared__ PrunedShared sh;
  const LinkParams &p = pp.lp;
  if (sweep_dead(p.ctl)) return;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long nrec = p.rec_ptr[p.P];
  for (long long ridx = (long long)blockIdx.x * LINK_WARPS + warp; ridx < nrec; ridx += (long long)gridDim.x * LINK_WARPS) {
    pruned_record(pp, sh, ridx, warp, lane);
    __syncwarp();  // the warp's shared tables are rewritten by the next record
  }
}

// The records k_link_pruned left aside, one CTA each: the warps share out the chunks of the block (a chunk's lane sums
// only depend on the chunk), warp 0 accumulates the check-points in chunk order and finishes the draw from the stored
// sums -- the same numbers, operation for operation, as one warp walking the block.
__global__ void __launch_bounds__(HEAVY_WARPS * 32) k_link_heavy(PrunedParams pp) {
  __shared__ RecAttr s_ra[DBL_MAX_ATTRS];
  __shared__ double s_sums[32 * 32];
  const LinkParams &p = pp.lp;
  if (sweep_dead(p.ctl)) return;
  const int nh = (int)p.ctl[CTL_HEAVY];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int A = p.A;
  for (int h = blockIdx.x; h < nh; h += gridDim.x) {
    const int ridx = pp.heavy_list[h];
    const int r = p.rec_sorted[ridx];
    const int b = pp.rec_key_sorted[ridx] >> pp.rec_key_shift;
    const int n = p.ent_ptr[b + 1] - p.ent_ptr[b];
    const int ntiles = p.tile_ptr[b + 1] - p.tile_ptr[b];
    const size_t tw = tile_words(A);
    const int *tiles = p.tiles + (size_t)p.tile_ptr[b] * tw;
    __syncthreads();  // the previous record's tables and sums are no longer read
    if (warp == 0 && lane < A) {
      RecAttr c;
      prep_rec_attr(p, r, lane, c);
      s_ra[lane] = c;
    }
    __syncthreads();
    const int nsteps = ntiles * (TE / 32);
    const int spc = (TE / 32) * max(1, (ntiles + 31) >> 5);
    const int nchunks = (nsteps + spc - 1) / spc;
    auto wf = [&](int j) -> double {
      if (j >= n) return 0.0;
      const int *tile = tiles + (size_t)(j / TE) * tw;
      const int slot = j % TE;
      return generic_weight(s_ra, A, false, tile + slot, reinterpret_cast<const double *>(tile + (size_t)A * TE)[slot]);
    };
    for (int c = warp; c < nchunks; c += HEAVY_WARPS) {
      double acc = 0.0;
      const int s1 = min((c + 1) * spc, nsteps);
      for (int st = c * spc; st < s1; ++st) acc = acc + wf((st << 5) + lane);
      s_sums[c * 32 + lane] = acc;
    }
    __syncthreads();
    if (warp == 0) {
      double run = 0.0, Q = 0.0;
      for (int c = 0; c < nchunks; ++c) {
        run = run + butterfly_sum(s_sums[c * 32 + lane]);
        if (lane == c) Q = run;
      }
      if (!(run > 0.0) || isinf(run)) {
        fail_link(p, lane, r);
      } else {
        const U2 u = uniform2(p.seed, PH_LINK, link_iter(p), (uint32_t)r, 0u);
        const int j = finish_draw(lane, n, nsteps, spc, nchunks, Q, run, u.u0, wf, s_sums);
        store_link(p, lane, r, b, n, j);
      }
    }
  }
}
#endif  // DBL_ENGINE_TU
