// Device half of libdblink_b200: the Gibbs sweep of dblink's record-linkage model on one B200.
//
// Reference (cleanzr/dblink @ dc3dd0d, src/main/scala/com/github/cleanzr/dblink/, GU = GibbsUpdates.scala):
//   State.nextState State.scala:78-99 -> updatePartition GU:156-211
//     link draw per record        GU:363-395 (PCG-II), GU:399-466 (PCG-I / Gibbs, dense form)   -> k_link
//     entity values per (e, attr) GU:534-599, 605-646, 702-755                                   -> k_values
//     distortions per (r, attr)   GU:324-359                                                     -> k_dist
//     new partition id            GU:206, partitioning/MutableBST.scala:61-79                    -> k_entity_post
//   updateSummaryVariables GU:219-301                                   -> k_entity_post / k_dist accumulators
//   the shuffle GU:144                                                  -> relayout() (sort by block id)
//
// Numerics: all likelihood arithmetic is IEEE binary64 with no FMA contraction (-fmad=false) so that the
// CPU oracle (oracle/dbl_oracle.c, -ffp-contract=off) reproduces every draw bit for bit.  Draw protocol:
// DESIGN.md section 4.
#include <cuda_runtime.h>
#include <unistd.h>

#include <algorithm>
#include <cfloat>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <cub/cub.cuh>
#include <map>
#include <string>
#include <vector>

#include "dbl_internal.h"
#define DBL_ENGINE_TU 1
#include "dbl_link.cuh"
#include "dbl_link_pcg2.cuh"

#define CUDA_TRY(expr)                                                                          \
  do {                                                                                          \
    cudaError_t _e = (expr);                                                                    \
    if (_e != cudaSuccess) {                                                                    \
      ctx->set_error(std::string(#expr) + ": " + cudaGetErrorString(_e));                       \
      return DBL_ERR_CUDA;                                                                      \
    }                                                                                           \
  } while (0)

// ---------------------------------------------------------------------------------------------------
// device-side model
// ---------------------------------------------------------------------------------------------------
struct TreeDev {
  int n_nodes;
  const int *attr, *kind, *split, *set_ptr, *set_val, *leaf_no;
};

// ---------------------------------------------------------------------------------------------------
// small helpers
// ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ int invcdf(const double *cdf, int V, double u) {
  int lo = 0, hi = V;
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (cdf[mid] > u) hi = mid; else lo = mid + 1;
  }
  return lo < V ? lo : V - 1;
}

__device__ __forceinline__ int tree_leaf(const TreeDev &t, const int *yrow) {
  int node = 0;
  while (node < t.n_nodes && t.attr[node] >= 0) {
    const int v = yrow[t.attr[node]];
    bool right;
    if (t.kind[node]) {
      int lo = t.set_ptr[node], hi = t.set_ptr[node + 1] - 1;
      right = false;
      while (lo <= hi) {
        const int mid = (lo + hi) >> 1;
        const int s = t.set_val[mid];
        if (s == v) { right = true; break; }
        if (s < v) lo = mid + 1; else hi = mid - 1;
      }
    } else {
      right = v > t.split[node];
    }
    node = right ? 2 * node + 2 : 2 * node + 1;
  }
  return t.leaf_no[node];
}

// ---------------------------------------------------------------------------------------------------
// Row kernels run in one of two modes:
//   prefix mode (inside a sweep): rows = the first ctl[CTL_OWNED_*] entries of ent_sorted / rec_sorted, i.e. exactly
//     the entities / records of the blocks this rank owns, counted on the DEVICE (no host round trip); grid-stride,
//     so the launch does not depend on the count; the kernel returns at once when the sweep was abandoned;
//   mask mode (state set-up): every row whose ownership byte is set.
// ---------------------------------------------------------------------------------------------------
struct RowSet {
  const long long *ctl;         // control block
  const int *sorted;            // ent_sorted / rec_sorted (prefix mode) or nullptr (mask mode)
  const unsigned char *owned;   // ownership bytes (mask mode)
  int64_t n_all;                // E or R
  int count_word;               // CTL_OWNED_ENT / CTL_OWNED_REC
  __device__ __forceinline__ int64_t count() const { return sorted ? (int64_t)ctl[count_word] : n_all; }
  __device__ __forceinline__ int64_t row(int64_t i) const {
    if (sorted) return sorted[i];
    return owned[i] ? i : -1;
  }
  __device__ __forceinline__ bool dead() const { return sorted && sweep_dead(ctl); }
};
#define GRID_STRIDE(i, n) \
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < (n); i += (int64_t)gridDim.x * blockDim.x)

// one atomic per distinct key among the active lanes of the warp
__device__ __forceinline__ void warp_hist_add(unsigned long long *bins, int key) {
  const unsigned peers = __match_any_sync(__activemask(), key);
  if ((__ffs(peers) - 1) == (int)(threadIdx.x & 31)) atomicAdd(&bins[key], (unsigned long long)__popc(peers));
}

// ---------------------------------------------------------------------------------------------------
// k_entity_post: per entity N(e) = prod_{non-const a} n_a(y_a); new block id (GU:206); entity part of the
// summary: isolates (GU:267-269) and sum_a log phi_a(y_a) (GU:234-237, 271-274); sizes of the new blocks (the
// input of the block -> rank placement, partitioning/LPTScheduler.scala:57-76).
// part = partial summary words of this rank: [A*F] aggDist, [A+1] recDist, isolates, log-likelihood (f64 bits),
// [P] entities per block, [P] records per block.
// ---------------------------------------------------------------------------------------------------
struct EntPostParams {
  RowSet rows;
  int A;
  const int *y;
  const AttrDev *attrs;
  TreeDev tree;
  double *entN;
  int *blk;
  const int *ent_rec_ptr;  // nullptr: no summary
  unsigned long long *part;
  int iso_slot, ll_slot, blk_slot;  // blk_slot < 0: no block histogram
};
__global__ void __launch_bounds__(256) k_entity_post(EntPostParams p) {
  if (p.rows.dead()) return;
  const int64_t n = p.rows.count();
  double ll = 0.0;
  int iso = 0;
  GRID_STRIDE(i, n) {
    const int64_t e = p.rows.row(i);
    if (e < 0) continue;
    const int *ye = p.y + e * p.A;
    double nn = 1.0;
    for (int a = 0; a < p.A; ++a) {
      const AttrDev &at = p.attrs[a];
      const int v = ye[a];
      if (!at.is_const) nn = nn * at.norm[v];
      ll += at.logphi[v];
    }
    p.entN[e] = nn;
    const int b = p.tree.n_nodes > 0 ? tree_leaf(p.tree, ye) : 0;
    p.blk[e] = b;
    if (p.ent_rec_ptr) {
      iso += (p.ent_rec_ptr[e] == p.ent_rec_ptr[e + 1]);
      if (p.blk_slot >= 0) warp_hist_add(p.part + p.blk_slot, b);
    }
  }
  if (p.ent_rec_ptr) {
    typedef cub::BlockReduce<double, 256> BR;
    typedef cub::BlockReduce<int, 256> BRI;
    __shared__ typename BR::TempStorage t1;
    __shared__ typename BRI::TempStorage t2;
    const double s = BR(t1).Sum(ll);
    const int c = BRI(t2).Sum(iso);
    if (threadIdx.x == 0) {
      if (s != 0.0) atomicAdd(reinterpret_cast<double *>(&p.part[p.ll_slot]), s);
      if (c) atomicAdd(&p.part[p.iso_slot], (unsigned long long)c);
    }
  }
}

// ---------------------------------------------------------------------------------------------------
// layout ("re-partitioning", replaces the shuffle GU:144): entities and records grouped by block
// ---------------------------------------------------------------------------------------------------
__global__ void k_iota(int64_t n, int *out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = (int)i;
}
__global__ void k_hist(int64_t n, const int *__restrict__ key, int *__restrict__ cnt) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) atomicAdd(&cnt[key[i]], 1);
}
// sort keys; entities / records this rank does not own go to the dummy slot (block P, entity E)
// Records are grouped by block and, within a block, by a static cost class, so that the records sharing a CTA of
// the link kernel (and its tile ring) advance at the same pace.  The order of records inside a block has no effect
// on the draws (every record has its own counter-based stream).
constexpr int REC_CLASS_BITS = 8;
// cost class of a record (x is static): bits 7..6 = number of missing non-constant attributes (each one adds a
// gather per candidate), bits 5..0 = expected number of similar-but-different candidate values per 32-candidate
// step (how often the warp takes the rare multiply: equal or similar value), from the empirical value frequencies.
__global__ void k_rec_class(int64_t R, int A, const AttrDev *__restrict__ attrs, const int *__restrict__ x,
                            unsigned char *__restrict__ cls) {
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= R) return;
  int miss = 0;
  double h = 0.0;
  for (int a = 0; a < A; ++a) {
    const AttrDev &at = attrs[a];
    if (at.is_const) continue;
    const int xv = x[r * A + a];
    if (xv < 0) { ++miss; continue; }
    h += at.probs[xv];  // an equal value takes the same path as a similar one (one table, see k_link_pcg2)
    for (int i = at.rowptr[xv]; i < at.rowptr[xv + 1]; ++i)
      if (at.col[i] != xv) h += at.probs[at.col[i]];
  }
  const int hq = min(63, (int)(h * 32.0 * 8.0));
  cls[r] = (unsigned char)((min(miss, 3) << 6) | hq);
}
// block sort keys of the entities and of the records in one launch
__global__ void k_block_keys(int64_t E, int64_t R, const int *__restrict__ blk, const int *__restrict__ link,
                             const unsigned char *__restrict__ ent_owned, const unsigned char *__restrict__ rec_owned,
                             const unsigned char *__restrict__ rec_class, int P, int *__restrict__ ent_key,
                             int *__restrict__ rec_key) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < E) ent_key[i] = ent_owned[i] ? blk[i] : P;
  if (i < R)  // not owned: behind every owned key, spread over the class bits (see sentinel_spread)
    rec_key[i] = rec_owned[i] ? ((blk[link[i]] << REC_CLASS_BITS) | rec_class[i])
                              : ((P << REC_CLASS_BITS) | (int)(i & ((1 << REC_CLASS_BITS) - 1)));
}
__global__ void k_rec_link_keys(int64_t R, const int *__restrict__ link, const unsigned char *__restrict__ rec_owned,
                                int E, int spread, int *__restrict__ key) {
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r < R) key[r] = rec_owned[r] ? link[r] : E + (int)(r % spread);  // see sentinel_spread
}
// the same inside a sweep, fused with the commit of the link draws: the link kernels wrote them to newlink; they
// become the state only if no categorical of the sweep was without mass (the reference fails the task and no new
// state exists, IndexNonUniformDiscreteDist.scala:78-79)
__global__ void k_commit_link_keys(int64_t R, const long long *__restrict__ ctl, const int *__restrict__ newlink,
                                   int *__restrict__ link, const unsigned char *__restrict__ rec_owned, int E,
                                   int spread, int *__restrict__ key) {
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= R) return;
  int l = link[r];
  const bool own = rec_owned[r];
  if (own && !sweep_dead(ctl)) {
    l = newlink[r];
    link[r] = l;
  }
  key[r] = own ? l : E + (int)(r % spread);  // see sentinel_spread
}
// offsets from sorted keys: ptr[k] = first position whose key is >= k, for k = 0..n_keys (keys beyond the data
// point at n).  One pass over the sorted array; replaces an atomic histogram + scan.
__device__ __forceinline__ void segment_ptr_at(int64_t i, int64_t n, int n_keys, const int *__restrict__ sorted_key,
                                               int *__restrict__ ptr, int shift) {
  if (i > n) return;
  const int cur = (i < n) ? min(sorted_key[i] >> shift, n_keys) : n_keys;
  const int prev = (i > 0) ? min(sorted_key[i - 1] >> shift, n_keys) : -1;
  for (int k = prev + 1; k <= cur; ++k) ptr[k] = (int)i;
}
__global__ void k_segment_ptr(int64_t n, int n_keys, const int *__restrict__ sorted_key, int *__restrict__ ptr,
                              int shift = 0) {
  segment_ptr_at((int64_t)blockIdx.x * blockDim.x + threadIdx.x, n, n_keys, sorted_key, ptr, shift);
}
// block offsets of the sorted entities and of the sorted records in one launch
__global__ void k_block_ptrs(int64_t E, int64_t R, int P, const int *__restrict__ blk_sorted, int *__restrict__ ent_ptr,
                             const int *__restrict__ rec_key_sorted, int *__restrict__ rec_ptr) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  segment_ptr_at(i, E, P, blk_sorted, ent_ptr, 0);
  segment_ptr_at(i, R, P, rec_key_sorted, rec_ptr, REC_CLASS_BITS);
}
// prefix sums over the P blocks (P is 2^numLevels: small); publishes the owned counts (everything before the dummy
// block) in the control block -- they size the prefix-mode row kernels of the next sweep.  As the last kernel of a
// sweep it also adopts the partial summary as the global one (single rank: adopt_nw > 0) and counts the sweep
// (finish), unless the sweep was abandoned.
__global__ void k_block_scan(int P, const int *__restrict__ ent_ptr, const int *__restrict__ rec_ptr,
                             int *__restrict__ tile_ptr, int *__restrict__ cta_ptr, int warps_per_cta,
                             int *__restrict__ cta_ptr2, int warps_per_cta2, int *__restrict__ cta_ptr3,
                             int recs_per_item3, long long *__restrict__ ctl,
                             int adopt_nw, const unsigned long long *__restrict__ part, long long *__restrict__ glob,
                             int finish) {
  const bool dead = sweep_dead(ctl);
  if (adopt_nw > 0 && !dead)
    for (int i = threadIdx.x; i < adopt_nw; i += blockDim.x) glob[i] = (long long)part[i];
  if (threadIdx.x == 0) {
    int t = 0, c = 0, c2 = 0, c3 = 0;
    for (int b = 0; b < P; ++b) {
      tile_ptr[b] = t; cta_ptr[b] = c; cta_ptr2[b] = c2; cta_ptr3[b] = c3;
      t += (ent_ptr[b + 1] - ent_ptr[b] + TE - 1) / TE;
      const int nr = rec_ptr[b + 1] - rec_ptr[b];
      c += (nr + warps_per_cta - 1) / warps_per_cta;
      c2 += (nr + warps_per_cta2 - 1) / warps_per_cta2;
      c3 += (nr + recs_per_item3 - 1) / recs_per_item3;
    }
    tile_ptr[P] = t; cta_ptr[P] = c; cta_ptr2[P] = c2; cta_ptr3[P] = c3;
    ctl[CTL_OWNED_ENT] = ent_ptr[P];
    ctl[CTL_OWNED_REC] = rec_ptr[P];
    if (finish && !dead) ctl[CTL_ITER] += 1;
  }
}
// Tiled, block-sorted copies of the entity table, one thread per tile slot (padding slots of a block's last tile are
// zeroed here: no memset of the whole table).  fmt 1: attribute-major tiles { int32 y[A][TE]; f64 N[TE]; uint32
// packed_consts[TE] } (k_link_generic / k_link_match / k_link_pruned); fmt 2: quad tiles (k_link_pcg2).
__global__ void k_build_tiles(int64_t n_slots, int fmt, int A, const int *__restrict__ y, const double *__restrict__ entN,
                              const int *__restrict__ ent_sorted, const int *__restrict__ ent_ptr,
                              const int *__restrict__ tile_ptr, int *__restrict__ tiles, const int *__restrict__ perm, int P,
                              int npack, int *__restrict__ qtiles, int n_str, int qtile_pk) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_slots) return;
  const int T = (int)(i / TE), slot = (int)(i % TE);
  if (T >= tile_ptr[P]) return;
  int lo = 0, hi = P;  // block of tile T: last b with tile_ptr[b] <= T
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if (tile_ptr[mid] <= T) lo = mid; else hi = mid;
  }
  const int b = lo;
  const int j = (T - tile_ptr[b]) * TE + slot;
  const bool real = j < ent_ptr[b + 1] - ent_ptr[b];
  const int64_t e = real ? ent_sorted[ent_ptr[b] + j] : 0;
  unsigned pk = 0;  // constant attributes (kernel positions 0..npack-1), one byte each, for k_link_pcg2
  if (real)
    for (int k = 0; k < npack; ++k) pk |= ((unsigned)y[e * A + perm[k]] & 0xFFu) << (8 * k);
  const double nn = real ? entN[e] : 0.0;
  if (fmt == 1) {
    int *tile = tiles + (size_t)T * tile_words(A);
    for (int k = 0; k < A; ++k) tile[k * TE + slot] = real ? y[e * A + perm[k]] : 0;  // kernel order
    reinterpret_cast<double *>(tile + (size_t)A * TE)[slot] = nn;
    tile[(size_t)(A + 2) * TE + slot] = (int)pk;
  } else {
    const int nv = qtile_nv(A, n_str, qtile_pk != 0), ng = qtile_groups(nv), qw = qtile_words(nv);
    int *qt = qtiles + (size_t)T * qw * TE;
    int v[4];
    for (int g = 0; g < ng; ++g) {
      for (int c = 0; c < 4; ++c) {
        const int w = 4 * g + c;
        int val = 0;
        if (real) {
          if (qtile_pk) val = (w < n_str) ? y[e * A + perm[A - n_str + w]] : (w == n_str ? (int)pk : 0);
          else val = (w < A) ? y[e * A + perm[w]] : 0;
        }
        v[c] = val;
      }
      reinterpret_cast<int4 *>(qt)[(size_t)g * TE + slot] = make_int4(v[0], v[1], v[2], v[3]);
    }
    reinterpret_cast<double *>(qt + (size_t)ng * 4 * TE)[slot] = nn;
  }
}

// ---------------------------------------------------------------------------------------------------
// sweep bookkeeping on the device (the host only enqueues): theta draw, link commit, end of sweep
// ---------------------------------------------------------------------------------------------------
// updateDistProbs GU:305-320: theta[a,f] ~ Beta(alpha_a + aggDist[a,f], beta_a + N_f - aggDist[a,f]) from the GLOBAL
// summary of the previous state.  Every rank draws the same values from the same counter-based stream (replaces
// the broadcast, State.scala:84).  theta_prev keeps the old values: an abandoned sweep restores them.
__global__ void k_theta(int A, int F, uint64_t seed, long long *__restrict__ ctl, const long long *__restrict__ glob,
                        const double *__restrict__ alpha, const double *__restrict__ beta,
                        const double *__restrict__ file_size, double *__restrict__ theta,
                        double *__restrict__ theta_prev, unsigned long long *__restrict__ part, int nw) {
  if (sweep_dead(ctl)) return;
  for (int i = threadIdx.x; i < nw; i += blockDim.x) part[i] = 0ull;  // the partial summary of the sweep starts empty
  const uint32_t it = (uint32_t)(ctl[CTL_ITER] + 1);
  for (int i = threadIdx.x; i < A * F; i += blockDim.x) {
    const int a = i / F, f = i % F;
    theta_prev[i] = theta[i];
    theta[i] = draw_theta_one(seed, it, (uint32_t)i, alpha[a], beta[a], (double)glob[i], file_size[f]);
  }
  if (threadIdx.x == 0) { ctl[CTL_MOVED_ENT] = 0; ctl[CTL_MOVED_REC] = 0; ctl[CTL_WORK] = 0; ctl[CTL_HEAVY] = 0; }
}
// single rank: the partial summary is the global one
__global__ void k_reduce_local(int nw, const long long *__restrict__ ctl, const unsigned long long *__restrict__ part,
                               long long *__restrict__ glob) {
  if (sweep_dead(ctl)) return;
  for (int i = threadIdx.x; i < nw; i += blockDim.x) glob[i] = (long long)part[i];
}
__global__ void k_finish(long long *__restrict__ ctl) {
  if (threadIdx.x == 0 && !sweep_dead(ctl)) ctl[CTL_ITER] += 1;
}

// ---------------------------------------------------------------------------------------------------
// k_values: one thread per (entity, attribute).  updateEntityValueCollapsed GU:576-599 +
// perturbedDistYCollapsed GU:534-570 (PCG-I/II); updateEntityValue GU:605-646 + perturbedDistY GU:702-727.
// ---------------------------------------------------------------------------------------------------
// batched loads of k_values on sizes that fill the GPU (see value_update): value phase of a 1M sweep 1.129 ms with
// none (1), 1.089 with pairs (2), 1.151 with four at a time (64 registers either way: the spills grow)
#ifndef DBL_VALUES_UB_LARGE
#define DBL_VALUES_UB_LARGE 2
#endif
struct ValParams {
  int A, F, sampler;
  uint64_t seed;
  RowSet rows;  // owned entities
  const AttrDev *attrs;
  const int *x, *file;
  const unsigned *zmask;
  const double *theta;
  const int *ent_rec_ptr, *rec_by_ent;
  int *y;
};

struct BaseDist {
  const AttrDev *at;
  int k;
  const double *pk, *cdf;
  double zk;
};
__device__ __forceinline__ double base_weight(const AttrDev &at, int k, int v) {
  double w = at.probs[v];
  if (!at.is_const)
    for (int i = 0; i < k; ++i) w = w * at.norm[v];
  return w;
}
__device__ void base_init(BaseDist &b, const AttrDev &at, int k) {
  b.at = &at;
  if (at.is_const) k = 0;
  b.k = k;
  if (k <= at.kmax) {
    b.pk = at.pk + (size_t)k * at.V;
    b.cdf = at.cdf + (size_t)k * at.V;
    b.zk = 0.0;
  } else {  // beyond the cached powers (getSimNormDist cache miss, AttributeIndex.scala:199-205)
    b.pk = nullptr; b.cdf = nullptr;
    double z = 0.0;
    for (int v = 0; v < at.V; ++v) z += base_weight(at, k, v);
    b.zk = z;
  }
}
__device__ __forceinline__ double base_prob(const BaseDist &b, int v) {
  return b.pk ? b.pk[v] : base_weight(*b.at, b.k, v) / b.zk;
}
__device__ int base_draw(const BaseDist &b, double u) {
  if (b.cdf) return invcdf(b.cdf, b.at->V, u);
  double c = 0.0;
  for (int v = 0; v < b.at->V; ++v) {
    c += base_weight(*b.at, b.k, v) / b.zk;
    if (c > u) return v;
  }
  return b.at->V - 1;
}

// factor contributed by record r to candidate value v; false when v is outside the record's support
__device__ __forceinline__ bool g_factor(const ValParams &p, const AttrDev &at, int a, int r, bool collapsed, int v,
                                         double &g) {
  const int xr = p.x[(int64_t)r * p.A + a];
  if (at.is_const) {
    if (v != xr || !collapsed) return false;
    const double th = p.theta[a * p.F + p.file[r]];
    g = 1.0 + (1.0 / th - 1.0) / at.phi[xr];  // GU:553
    return true;
  }
  double e;
  if (!row_find(at, xr, v, e)) return false;
  if (collapsed && v == xr) {
    const double th = p.theta[a * p.F + p.file[r]];
    g = e + (1.0 / th - 1.0) / (at.phi[xr] * at.norm[xr]);  // GU:557,560
  } else {
    g = e;
  }
  return true;
}
__device__ __forceinline__ bool in_support(const ValParams &p, const AttrDev &at, int a, int r, int v) {
  const int xr = p.x[(int64_t)r * p.A + a];
  if (at.is_const) return v == xr;
  double e;
  return row_find(at, xr, v, e);
}

constexpr int VALUE_REDO = -2;  // what k_values stores for a draw it leaves to k_values_log
// marks the running sweep for k_values_log in the control block (a word only these two kernels use; through the
// RowSet's pointer, since one more kernel parameter alone changes the register allocation of k_values)
__device__ __forceinline__ int redo_later(const ValParams &p, uint32_t iter) {
  const_cast<long long *>(p.rows.ctl)[CTL_VALUES_REDO] = iter;
  return VALUE_REDO;
}

// The mixture of GU:593-597 in the log domain (DESIGN.md 4.3), for the draws whose sum of perturbation weights is
// not finite: a large cluster of agreeing records overflows prod_r g_r(v), and beyond the cached powers n(v)^k can
// underflow to 0 / 0.  log b_k(v) = log probs(v) + k log n(v); log W(v) = log b_k(v) + log(G(v) - 1), or
// log b_k(v) + sum_r log g_r(v) where G itself overflows.  The same candidates in the same order as value_update,
// with det_log / det_exp, so the oracle draws the same value (oracle/dbl_oracle.c value_draw_log).
__device__ __noinline__ int value_update_log(const ValParams &p, const AttrDev &at, int a, int lo, int hi, int k,
                                             bool collapsed, U2 u) {
  const int *rec = p.rec_by_ent;
  const double kk = at.is_const ? 0.0 : (double)k;
  auto lbase = [&](int v) { return det_log(at.probs[v]) + kk * det_log(at.norm[v]); };
  double bmax = lbase(0), Z = 0.0;  // Z = sum_v b_k(v) / exp(bmax) over every value, in ascending id
  for (int v = 1; v < at.V; ++v) {
    const double l = lbase(v);
    if (l > bmax) bmax = l;
  }
  for (int v = 0; v < at.V; ++v) Z += det_exp(lbase(v) - bmax);
  // pass 0: max of log W; pass 1: sum of exp(log W - max); pass 2: the inverse CDF at u1
  double lmax = 0.0, S = 0.0, target = 0.0, cum = 0.0;
  bool any = false, base = false;
  int picked = -1, last_pos = -1;
  for (int pass = 0; pass < 3 && !base && picked < 0; ++pass) {
    for (int i = lo; i < hi && picked < 0; ++i) {
      const int xr = p.x[(int64_t)rec[i] * p.A + a];
      if (xr < 0) continue;
      bool repeated = false;  // every value of this record's row has been seen (value_update)
      for (int j = lo; j < i && !repeated; ++j) repeated = (p.x[(int64_t)rec[j] * p.A + a] == xr);
      if (repeated) continue;
      const int nv = at.is_const ? 1 : (at.rowptr[xr + 1] - at.rowptr[xr]);
      for (int q = 0; q < nv && picked < 0; ++q) {
        const int v = at.is_const ? xr : at.col[at.rowptr[xr] + q];
        bool seen = false;
        for (int j = lo; j < i && !seen; ++j) {
          const int rj = rec[j];
          if (p.x[(int64_t)rj * p.A + a] < 0) continue;
          seen = in_support(p, at, a, rj, v);
        }
        if (seen) continue;
        double G = 1.0, L = 0.0;
        for (int j = i; j < hi; ++j) {
          const int rj = rec[j];
          if (p.x[(int64_t)rj * p.A + a] < 0) continue;
          double g;
          if (g_factor(p, at, a, rj, collapsed, v, g)) { G = G * g; L = L + det_log(g); }
        }
        if (!(G > 1.0)) continue;  // W(v) = 0
        const double lw = lbase(v) + (G <= DBL_MAX ? det_log(G - 1.0) : L);
        if (pass == 0) {
          if (!any || lw > lmax) lmax = lw;
          any = true;
        } else if (pass == 1) {
          S += det_exp(lw - lmax);
        } else {
          const double W = det_exp(lw - lmax);
          cum += W;
          if (W > 0.0) last_pos = v;
          if (cum > target) picked = v;
        }
      }
    }
    if (pass == 0 && !any) base = true;
    if (pass == 1) {  // P(base) = Z / (Z + sum W)  (GU:593-594)
      const double d = (lmax + det_log(S)) - (bmax + det_log(Z));
      base = u.u0 < 1.0 / (1.0 + det_exp(d));
      target = u.u1 * S;
    }
  }
  if (!base) return picked >= 0 ? picked : last_pos;
  const double bt = u.u1 * Z;
  double c = 0.0;
  for (int v = 0; v < at.V; ++v) {
    c += det_exp(lbase(v) - bmax);
    if (c > bt) return v;
  }
  return at.V - 1;
}

// new value of attribute a of entity e.  UB > 1: the loop over the similarity row of a single linked record fetches
// UB candidates at a time (independent loads, same sums in the same order): for problems too small to fill the GPU
// the kernel's time is the longest dependent-load chain of one thread, not throughput
template <int UB>
__device__ int value_update(const ValParams &p, uint32_t iter, int64_t e, int a) {
  const AttrDev &at = p.attrs[a];
  const bool collapsed = (p.sampler == DBL_PCG_I || p.sampler == DBL_PCG_II);
  const U2 u = uniform2(p.seed, PH_VALUE, iter, (uint32_t)e, (uint32_t)a);
  const int lo = p.ent_rec_ptr[e], hi = p.ent_rec_ptr[e + 1];
  const int *rec = p.rec_by_ent;

  int k = 0;
  for (int i = lo; i < hi; ++i) k += (p.x[(int64_t)rec[i] * p.A + a] >= 0);
  BaseDist b;
  if (k == 0) {  // GU:588-589
    base_init(b, at, 0);
    return base_draw(b, u.u1);
  }
  if (!collapsed) {
    for (int i = lo; i < hi; ++i) {  // GU:619-630
      const int r = rec[i];
      const int xr = p.x[(int64_t)r * p.A + a];
      if (xr >= 0 && !((p.zmask[r] >> a) & 1u)) return xr;
    }
    if (at.is_const) {  // GU:633-634
      base_init(b, at, 0);
      return base_draw(b, u.u1);
    }
  }
  base_init(b, at, k);  // GU:584-586
  double total = 0.0, target = 0.0, cum = 0.0;
  int picked = -1, last_pos = -1;
  if (hi - lo == 1) {
    // one linked record (most entities): the candidate values are the record's own similarity row, so the factors
    // come straight from that row (no searches, no first-appearance check); same operations as the general path
    const int r = rec[lo];
    const int xr = p.x[(int64_t)r * p.A + a];  // observed (k == 1)
    const int q0 = at.is_const ? 0 : at.rowptr[xr];
    const int nv = at.is_const ? 1 : (at.rowptr[xr + 1] - q0);
    double extra = 0.0;  // what the collapsed update adds to the factor of v == x (GU:553,557,560)
    if (collapsed) {
      const double th = p.theta[a * p.F + p.file[r]];
      extra = at.is_const ? (1.0 / th - 1.0) / at.phi[xr] : (1.0 / th - 1.0) / (at.phi[xr] * at.norm[xr]);
    }
    auto weight = [&](int q, int &v) -> double {
      double G = 1.0;
      if (at.is_const) {
        v = xr;
        if (collapsed) G = G * (1.0 + extra);
      } else {
        v = at.col[q0 + q];
        const double ex = at.expsim[q0 + q];
        G = G * ((collapsed && v == xr) ? ex + extra : ex);
      }
      return base_prob(b, v) * (G - 1.0);  // GU:567 / 724
    };
    if constexpr (UB > 1) {
      // same weights, same order of the sums; the loads of UB consecutive candidates are issued together
      auto batch = [&](int q, int (&v)[UB], double (&W)[UB]) {
        double ex[UB], bp[UB];
#pragma unroll
        for (int i = 0; i < UB; ++i) {
          const int qq = min(q + i, nv - 1);
          v[i] = at.is_const ? xr : at.col[q0 + qq];
          ex[i] = at.is_const ? 0.0 : at.expsim[q0 + qq];
        }
#pragma unroll
        for (int i = 0; i < UB; ++i) bp[i] = base_prob(b, v[i]);
#pragma unroll
        for (int i = 0; i < UB; ++i) {
          double G = 1.0;
          if (at.is_const) { if (collapsed) G = G * (1.0 + extra); }
          else G = G * ((collapsed && v[i] == xr) ? ex[i] + extra : ex[i]);
          W[i] = bp[i] * (G - 1.0);
        }
      };
      for (int q = 0; q < nv; q += UB) {
        int v[UB];
        double W[UB];
        batch(q, v, W);
#pragma unroll
        for (int i = 0; i < UB; ++i)
          if (q + i < nv) total += W[i];
      }
      if (!isfinite(total)) return redo_later(p, iter);
      if (u.u0 < 1.0 / (1.0 + total)) return base_draw(b, u.u1);  // GU:593-594
      target = u.u1 * total;
      for (int q = 0; q < nv && picked < 0; q += UB) {
        int v[UB];
        double W[UB];
        batch(q, v, W);
#pragma unroll
        for (int i = 0; i < UB; ++i)
          if (q + i < nv && picked < 0) {
            cum += W[i];
            if (W[i] > 0.0) last_pos = v[i];
            if (cum > target) picked = v[i];
          }
      }
    } else {
      for (int q = 0; q < nv; ++q) {
        int v;
        total += weight(q, v);
      }
      if (!isfinite(total)) return redo_later(p, iter);
      if (u.u0 < 1.0 / (1.0 + total)) return base_draw(b, u.u1);  // GU:593-594
      target = u.u1 * total;
      for (int q = 0; q < nv && picked < 0; ++q) {
        int v;
        const double W = weight(q, v);
        cum += W;
        if (W > 0.0) last_pos = v;
        if (cum > target) picked = v;
      }
    }
    if (picked < 0) picked = last_pos;
    if (picked < 0) picked = base_draw(b, u.u1);
    return picked;
  }
  for (int pass = 0; pass < 2; ++pass) {
    for (int i = lo; i < hi; ++i) {
      const int r = rec[i];
      const int xr = p.x[(int64_t)r * p.A + a];
      if (xr < 0) continue;
      // an earlier record with the same value has already introduced every value of this record's similarity row
      // (the usual case inside a cluster: duplicates agree): nothing new to add, and no pairwise searches
      bool repeated = false;
      for (int j = lo; j < i && !repeated; ++j) repeated = (p.x[(int64_t)rec[j] * p.A + a] == xr);
      if (repeated) continue;
      const int nv = at.is_const ? 1 : (at.rowptr[xr + 1] - at.rowptr[xr]);
      const int *vals = at.is_const ? nullptr : (at.col + at.rowptr[xr]);
      for (int q = 0; q < nv; ++q) {
        const int v = at.is_const ? xr : vals[q];
        bool seen = false;
        for (int j = lo; j < i && !seen; ++j) {
          const int rj = rec[j];
          if (p.x[(int64_t)rj * p.A + a] < 0) continue;
          seen = in_support(p, at, a, rj, v);
        }
        if (seen) continue;
        double G = 1.0;
        for (int j = i; j < hi; ++j) {
          const int rj = rec[j];
          const int xj = p.x[(int64_t)rj * p.A + a];
          if (xj < 0) continue;
          double g;
          if (!at.is_const && xj == xr) {
            // a record observing the same value as record i (record i itself; duplicates that agree): v sits at
            // position q of that value's row, so the search of g_factor would return exactly this element
            const double ex = at.expsim[at.rowptr[xr] + q];
            if (collapsed && v == xr) {
              const double th = p.theta[a * p.F + p.file[rj]];
              g = ex + (1.0 / th - 1.0) / (at.phi[xr] * at.norm[xr]);  // GU:557,560
            } else {
              g = ex;
            }
            G = G * g;
          } else if (g_factor(p, at, a, rj, collapsed, v, g)) {
            G = G * g;
          }
        }
        const double W = base_prob(b, v) * (G - 1.0);  // GU:567 / 724
        if (pass == 0) {
          total += W;
        } else {
          cum += W;
          if (W > 0.0) last_pos = v;
          if (picked < 0 && cum > target) picked = v;
        }
      }
    }
    if (pass == 0) {
      if (!isfinite(total)) return redo_later(p, iter);
      if (u.u0 < 1.0 / (1.0 + total)) return base_draw(b, u.u1);  // GU:593-594
      target = u.u1 * total;
    }
  }
  if (picked < 0) picked = last_pos;
  if (picked < 0) picked = base_draw(b, u.u1);
  return picked;
}

template <int UB>
__global__ void __launch_bounds__(128) k_values(ValParams p) {
  if (p.rows.dead()) return;
  const uint32_t iter = (uint32_t)(p.rows.ctl[CTL_ITER] + 1);
  const int64_t n = p.rows.count() * p.A;
  GRID_STRIDE(t, n) {  // entity-major: the attributes of an entity share its record list (an attribute-major mapping,
                       // one code path per warp, measured slower: 1.11 vs 0.88 ms at 1M)
    const int64_t e = p.rows.row(t / p.A);
    if (e < 0) continue;
    const int a = (int)(t % p.A);
    p.y[e * p.A + a] = value_update<UB>(p, iter, e, a);
  }
}

// The draws k_values left (sum of the perturbation weights not finite), in the log domain.  A kernel of its own, so
// that the rarely taken fallback costs k_values nothing (registers, stack): when no draw was left in this sweep every
// block returns at once.
__global__ void __launch_bounds__(128) k_values_log(ValParams p) {
  if (p.rows.dead()) return;
  const uint32_t iter = (uint32_t)(p.rows.ctl[CTL_ITER] + 1);
  if (p.rows.ctl[CTL_VALUES_REDO] != (long long)iter) return;
  const bool collapsed = (p.sampler == DBL_PCG_I || p.sampler == DBL_PCG_II);
  const int64_t n = p.rows.count() * p.A;
  GRID_STRIDE(t, n) {
    const int64_t e = p.rows.row(t / p.A);
    if (e < 0) continue;
    const int a = (int)(t % p.A);
    if (p.y[e * p.A + a] != VALUE_REDO) continue;
    const int lo = p.ent_rec_ptr[e], hi = p.ent_rec_ptr[e + 1];
    int k = 0;
    for (int i = lo; i < hi; ++i) k += (p.x[(int64_t)p.rec_by_ent[i] * p.A + a] >= 0);
    const U2 u = uniform2(p.seed, PH_VALUE, iter, (uint32_t)e, (uint32_t)a);
    p.y[e * p.A + a] = value_update_log(p, p.attrs[a], a, lo, hi, k, collapsed, u);
  }
}

// ---------------------------------------------------------------------------------------------------
// k_dist: one thread per record.  updateDistortions GU:324-359 with the new y, fused with the record part
// of updateSummaryVariables GU:239-266.  draw = 0 only accumulates the summary of the current state.
// ---------------------------------------------------------------------------------------------------
struct DistParams {
  int A, F, draw;
  uint64_t seed;
  RowSet rows;  // owned records
  const AttrDev *attrs;
  const int *x, *file, *link, *y, *blk;
  unsigned *zmask;
  const double *theta;
  unsigned long long *part;  // [A*F] aggDist, then [A+1] recDist, ...
  int ll_slot, blk_slot;     // blk_slot < 0: no block histogram
};

__global__ void __launch_bounds__(256) k_dist(DistParams p) {
  if (p.rows.dead()) return;
  const uint32_t iter = (uint32_t)(p.rows.ctl[CTL_ITER] + 1);
  const int64_t n = p.rows.count();
  double ll = 0.0;
  GRID_STRIDE(i, n) {
    const int64_t r = p.rows.row(i);
    if (r < 0) continue;
    const int f = p.file[r];
    const int e = p.link[r];
    const int *ye = p.y + (int64_t)e * p.A;
    unsigned zm = p.zmask[r];
    int nd = 0;
    for (int a = 0; a < p.A; ++a) {
      const AttrDev &at = p.attrs[a];
      const int xv = p.x[r * p.A + a];
      const int yv = ye[a];
      bool z;
      if (p.draw) {
        const double th = p.theta[a * p.F + f];
        if (xv < 0) {
          const U2 u = uniform2(p.seed, PH_DIST, iter, (uint32_t)r, (uint32_t)a);
          z = u.u0 < th;  // GU:331-334
        } else if (xv != yv) {
          z = true;  // GU:352-354
        } else {
          const U2 u = uniform2(p.seed, PH_DIST, iter, (uint32_t)r, (uint32_t)a);
          double pr1 = th * at.phi[xv];
          if (!at.is_const) {
            pr1 = pr1 * at.norm[xv];
            pr1 = pr1 * at.diag[xv];
          }
          const double pr0 = 1.0 - th;
          const double den = pr1 + pr0;
          const double pz = (den != 0.0) ? pr1 / den : 0.0;  // GU:349-350
          z = u.u0 < pz;
        }
        zm = z ? (zm | (1u << a)) : (zm & ~(1u << a));
      } else {
        z = (zm >> a) & 1u;
      }
      if (z) {
        ++nd;
        atomicAdd(&p.part[a * p.F + f], 1ull);  // GU:246
        if (xv >= 0) {                          // GU:248-258
          ll += at.logphi[xv];
          if (!at.is_const) {
            ll += at.lognorm[yv];
            double ex;
            if (row_find(at, xv, yv, ex)) ll += log(ex);
          }
        }
      }
    }
    if (p.draw) p.zmask[r] = zm;
    warp_hist_add(p.part + p.A * p.F, nd);  // GU:265
    if (p.blk_slot >= 0) warp_hist_add(p.part + p.blk_slot, p.blk[e]);
  }
  typedef cub::BlockReduce<double, 256> BR;
  __shared__ typename BR::TempStorage tmp;
  const double s = BR(tmp).Sum(ll);
  if (threadIdx.x == 0 && s != 0.0) atomicAdd(reinterpret_cast<double *>(&p.part[p.ll_slot]), s);
}

// ---------------------------------------------------------------------------------------------------
// k_init_state: State.deterministic (State.scala:253-301) -- entity e copies record e (if any), missing
// values drawn from phi; record r links to entity r mod E; z = (x>=0 && x!=y).
// ---------------------------------------------------------------------------------------------------
__global__ void k_init_entities(int64_t E, int64_t R, int A, uint64_t seed, const AttrDev *__restrict__ attrs,
                                const int *__restrict__ x, int *__restrict__ y) {
  const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (tid >= E * A) return;
  const int64_t e = tid / A;
  const int a = (int)(tid % A);
  int v = (e < R) ? x[e * A + a] : -1;
  if (v < 0) {
    const U2 u = uniform2(seed, PH_INIT, 0u, (uint32_t)e, (uint32_t)a);
    v = invcdf(attrs[a].cdf, attrs[a].V, u.u1);
  }
  y[tid] = v;
}
__global__ void k_init_records(int64_t E, int64_t R, int A, const int *__restrict__ x, const int *__restrict__ y,
                               int *__restrict__ link, unsigned *__restrict__ zmask) {
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= R) return;
  const int64_t e = r % E;
  link[r] = (int)e;
  unsigned zm = 0;
  for (int a = 0; a < A; ++a) {
    const int xv = x[r * A + a];
    if (xv >= 0 && xv != y[e * A + a]) zm |= 1u << a;
  }
  zmask[r] = zm;
}
// range checks of an uploaded state (the reference would fail with ArrayIndexOutOfBounds / require):
// bit 0 record value id, bit 1 file id, bit 2 link, bit 3 entity value id
__global__ void k_validate(int64_t R, int64_t E, int A, int F, const AttrDev *__restrict__ attrs,
                           const int *__restrict__ x, const int *__restrict__ file, const int *__restrict__ link,
                           const int *__restrict__ y, int *__restrict__ flag) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  int bad = 0;
  if (i < R) {
    for (int a = 0; a < A; ++a) {
      const int v = x[i * A + a];
      if (v < -1 || v >= attrs[a].V) bad |= 1;
    }
    if (file[i] < 0 || file[i] >= F) bad |= 2;
    if (link && (link[i] < 0 || link[i] >= E)) bad |= 4;
  }
  if (y && i < E)
    for (int a = 0; a < A; ++a) {
      const int v = y[i * A + a];
      if (v < 0 || v >= attrs[a].V) bad |= 8;
    }
  if (bad) atomicOr(flag, bad);
}
__global__ void k_pack_z(int64_t R, int A, const uint8_t *__restrict__ z, unsigned *__restrict__ zmask) {
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= R) return;
  unsigned zm = 0;
  for (int a = 0; a < A; ++a) zm |= (z[r * A + a] ? 1u : 0u) << a;
  zmask[r] = zm;
}
__global__ void k_unpack_z(int64_t R, int A, const unsigned *__restrict__ zmask, uint8_t *__restrict__ z) {
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= R) return;
  const unsigned zm = zmask[r];
  for (int a = 0; a < A; ++a) z[r * A + a] = (zm >> a) & 1u;
}

// ---------------------------------------------------------------------------------------------------
// multi-GPU: ownership and the exchange of clusters whose new block belongs to another rank (replaces the
// shuffle `.partitionBy(partitioner)`, GU:144).  Messages: entity = [e, y_0..y_{A-1}], record = [r, e, zmask].
// ---------------------------------------------------------------------------------------------------
__global__ void k_mark_ent_owned(int64_t E, const int *__restrict__ blk, const int *__restrict__ owner, int rank,
                                 unsigned char *__restrict__ ent_owned) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e < E) ent_owned[e] = (owner[blk[e]] == rank);
}
__global__ void k_mark_ent_block(int64_t E, const int *__restrict__ blk, int block, unsigned char *__restrict__ ent_owned) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e < E) ent_owned[e] = (blk[e] == block);
}
__global__ void k_mark_rec_owned(int64_t R, const int *__restrict__ link, const unsigned char *__restrict__ ent_owned,
                                 unsigned char *__restrict__ rec_owned) {
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r < R) rec_owned[r] = ent_owned[link[r]];
}

// ---- (1) peer-to-peer exchange: the data plane of a sharded dbl_sweep ---------------------------------------
// Every rank owns one communication buffer (cudaMalloc, exported with cudaIpc, mapped by every peer over
// NVLink/NVSwitch).  The kernels that decide which clusters leave write the messages STRAIGHT into the destination
// rank's receive buffer (slot from a system-scope atomic on the destination's cursor), the partial summary goes into
// a slot of every peer, one flag barrier follows, then every rank unpacks what it received and reduces the summary
// slots in rank order.  No host round trip, no separate pack / count / send / receive steps.  Receive buffers have
// room for EVERY entity and record (an entity moves at most once per sweep), and everything is double buffered by
// barrier parity, so a fast rank can run ahead by one sweep without overwriting what a slow one still reads.
constexpr int MAX_WORLD = 16;
struct CommDev {
  int rank, world, A, nws;  // nws = summary words per slot (partial summary + status)
  long long cap_e, cap_r;
  unsigned char *base[MAX_WORLD];  // communication buffer of every rank (own buffer at [rank])
  size_t off_cursor, off_slots, off_ent, off_rec;
  __device__ __forceinline__ unsigned long long *arrive(int d) const { return reinterpret_cast<unsigned long long *>(base[d]); }
  __device__ __forceinline__ unsigned long long *cursor(int d, int par) const {
    return reinterpret_cast<unsigned long long *>(base[d] + off_cursor) + 2 * par;
  }
  __device__ __forceinline__ long long *slot(int d, int par, int src) const {
    return reinterpret_cast<long long *>(base[d] + off_slots) + ((size_t)par * world + src) * nws;
  }
  __device__ __forceinline__ int *recv_ent(int d, int par) const {
    return reinterpret_cast<int *>(base[d] + off_ent) + (size_t)par * cap_e * (A + 1);
  }
  __device__ __forceinline__ int *recv_rec(int d, int par) const {
    return reinterpret_cast<int *>(base[d] + off_rec) + (size_t)par * cap_r * 3;
  }
};
__device__ __forceinline__ int comm_parity(const long long *ctl) { return (int)((ctl[CTL_EPOCH] + 1) & 1); }

// slot in rank d's buffer for every lane that has a message for d: one system-scope atomic per destination and warp.
// Every lane of the warp calls it (d < 0: nothing to send).
__device__ __forceinline__ long long remote_slot(unsigned long long *const *cursors_unused, const CommDev &c, int par,
                                                 int which, int d) {
  (void)cursors_unused;
  const int lane = threadIdx.x & 31;
  const unsigned grp = __match_any_sync(FULL, d);
  const int leader = __ffs(grp) - 1;
  unsigned long long basev = 0;
  if (d >= 0 && lane == leader) basev = atomicAdd_system(c.cursor(d, par) + which, (unsigned long long)__popc(grp));
  basev = __shfl_sync(FULL, basev, leader);
  return (long long)basev + __popc(grp & ((1u << lane) - 1u));
}

struct MoveParams {
  CommDev c;
  long long *ctl;
  int A;
  const int *ent_sorted, *rec_sorted;
  const int *blk, *owner, *link, *y;
  const unsigned *zmask;
  int *ent_dest;
  unsigned char *ent_owned, *rec_owned;
};
__global__ void __launch_bounds__(256) k_move_ent(MoveParams p) {
  if (sweep_dead(p.ctl)) return;
  const int64_t n = p.ctl[CTL_OWNED_ENT];
  const int64_t n32 = (n + 31) & ~(int64_t)31;  // whole warps stay in the loop together
  const int par = comm_parity(p.ctl);
  int sent = 0;
  GRID_STRIDE(i, n32) {
    int d = -1;
    int64_t e = -1;
    if (i < n) {
      e = p.ent_sorted[i];
      const int o = p.owner[p.blk[e]];
      if (o != p.c.rank) d = o;
      p.ent_dest[e] = d;
    }
    const long long slot = remote_slot(nullptr, p.c, par, 0, d);
    if (d >= 0) {
      int *m = p.c.recv_ent(d, par) + slot * (p.A + 1);
      m[0] = (int)e;
      for (int a = 0; a < p.A; ++a) m[1 + a] = p.y[e * p.A + a];
      p.ent_owned[e] = 0;
      ++sent;
    }
  }
  if (sent) atomicAdd(reinterpret_cast<unsigned long long *>(&p.ctl[CTL_MOVED_ENT]), (unsigned long long)sent);
}
__global__ void __launch_bounds__(256) k_move_rec(MoveParams p) {
  if (sweep_dead(p.ctl)) return;
  const int64_t n = p.ctl[CTL_OWNED_REC];
  const int64_t n32 = (n + 31) & ~(int64_t)31;
  const int par = comm_parity(p.ctl);
  int sent = 0;
  GRID_STRIDE(i, n32) {
    int d = -1;
    int64_t r = -1;
    if (i < n) {
      r = p.rec_sorted[i];
      d = p.ent_dest[p.link[r]];
    }
    const long long slot = remote_slot(nullptr, p.c, par, 1, d);
    if (d >= 0) {
      int *m = p.c.recv_rec(d, par) + slot * 3;
      m[0] = (int)r; m[1] = p.link[r]; m[2] = (int)p.zmask[r];
      p.rec_owned[r] = 0;
      ++sent;
    }
  }
  if (sent) atomicAdd(reinterpret_cast<unsigned long long *>(&p.ctl[CTL_MOVED_REC]), (unsigned long long)sent);
}
// partial summary (+ status) into a slot of every rank, then the barrier: rank r stores the new epoch into
// arrive[r] of every peer (release, system scope) and waits until its own arrive[] shows every peer (acquire).
// Never skipped, even when the sweep was abandoned locally: the peers are waiting.  A peer that does not show up
// within timeout_cycles sets ST_PEER_TIMEOUT instead of hanging the GPU.
__global__ void __launch_bounds__(256) k_publish_barrier(CommDev c, long long *ctl, const unsigned long long *part, int nw,
                                                         long long timeout_cycles) {
  const long long epoch = ctl[CTL_EPOCH] + 1;
  const int par = (int)(epoch & 1);
  __shared__ int s_timeout;
  if (threadIdx.x == 0) s_timeout = 0;
  for (int i = threadIdx.x; i < c.nws; i += blockDim.x) {
    const long long v = (i < nw) ? (long long)part[i] : ctl[CTL_STATUS];
    for (int d = 0; d < c.world; ++d) c.slot(d, par, c.rank)[i] = v;
  }
  __syncthreads();
  if ((int)threadIdx.x < c.world) {
    const int d = threadIdx.x;
    __threadfence_system();
    unsigned long long *flag = c.arrive(d) + c.rank;
    asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(flag), "l"((unsigned long long)epoch) : "memory");
    const unsigned long long *mine = c.arrive(c.rank) + d;
    const long long t0 = clock64();
    for (;;) {
      unsigned long long v;
      asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(mine) : "memory");
      if (v >= (unsigned long long)epoch) break;
      if (clock64() - t0 > timeout_cycles) { s_timeout = 1; break; }
      __nanosleep(200);
    }
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    ctl[CTL_EPOCH] = epoch;
    if (s_timeout) ctl[CTL_STATUS] |= ST_PEER_TIMEOUT;
  }
}
// what the peers wrote for this rank (parity of the barrier just passed)
__device__ __forceinline__ int done_parity(const long long *ctl) { return (int)(ctl[CTL_EPOCH] & 1); }
struct UnpackParams {
  CommDev c;
  const long long *ctl;
  int A;
  const AttrDev *attrs;
  TreeDev tree;
  int *y, *blk, *link;
  double *entN;
  unsigned *zmask;
  unsigned char *ent_owned, *rec_owned;
};
__global__ void __launch_bounds__(256) k_unpack_ent_p2p(UnpackParams p) {
  if (p.ctl[CTL_STATUS] & ST_PEER_TIMEOUT) return;
  const int par = done_parity(p.ctl);
  const int64_t n = (int64_t) * reinterpret_cast<volatile unsigned long long *>(p.c.cursor(p.c.rank, par));
  const int *buf = p.c.recv_ent(p.c.rank, par);
  GRID_STRIDE(i, n) {
    const int *m = buf + i * (p.A + 1);
    const int64_t e = m[0];
    double nn = 1.0;
    for (int a = 0; a < p.A; ++a) {
      const int v = m[1 + a];
      p.y[e * p.A + a] = v;
      if (!p.attrs[a].is_const) nn = nn * p.attrs[a].norm[v];
    }
    p.entN[e] = nn;
    p.blk[e] = p.tree.n_nodes > 0 ? tree_leaf(p.tree, m + 1) : 0;
    p.ent_owned[e] = 1;
  }
}
__global__ void __launch_bounds__(256) k_unpack_rec_p2p(UnpackParams p) {
  if (p.ctl[CTL_STATUS] & ST_PEER_TIMEOUT) return;
  const int par = done_parity(p.ctl);
  const int64_t n = (int64_t) * reinterpret_cast<volatile unsigned long long *>(p.c.cursor(p.c.rank, par) + 1);
  const int *buf = p.c.recv_rec(p.c.rank, par);
  GRID_STRIDE(i, n) {
    const int *m = buf + i * 3;
    const int64_t r = m[0];
    p.link[r] = m[1];
    p.zmask[r] = (unsigned)m[2];
    p.rec_owned[r] = 1;
  }
}
// global summary = sum of the slots in rank order (SummaryAccumulators.scala:54-63; integer words exact, the
// log-likelihood word is an f64 sum in a fixed order, so every rank gets identical bits); a peer's status makes the
// sweep fail here as well; the cursors of this parity are cleared for their next use two barriers from now
__global__ void __launch_bounds__(256) k_reduce_peers(CommDev c, long long *ctl, int nw, int ll_slot,
                                                      long long *__restrict__ glob) {
  const int par = done_parity(ctl);
  __shared__ long long s_status;
  if (threadIdx.x == 0) s_status = 0;
  __syncthreads();
  const bool timed_out = (ctl[CTL_STATUS] & ST_PEER_TIMEOUT) != 0;
  for (int i = threadIdx.x; i < c.nws && !timed_out; i += blockDim.x) {
    if (i == nw) {  // status word
      long long st = 0;
      for (int s = 0; s < c.world; ++s) st |= c.slot(c.rank, par, s)[i];
      if (st) atomicOr(reinterpret_cast<unsigned long long *>(&s_status), (unsigned long long)st);
    } else if (i == ll_slot) {
      double sum = 0.0;
      for (int s = 0; s < c.world; ++s) sum += __longlong_as_double(c.slot(c.rank, par, s)[i]);
      glob[i] = __double_as_longlong(sum);
    } else {
      long long sum = 0;
      for (int s = 0; s < c.world; ++s) sum += c.slot(c.rank, par, s)[i];
      glob[i] = sum;
    }
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    if (s_status && !ctl[CTL_STATUS]) ctl[CTL_STATUS] = (s_status & ST_ZERO_MASS) ? (ST_ZERO_MASS | ST_PEER_ERROR) : ST_PEER_ERROR;
    unsigned long long *cur = c.cursor(c.rank, par);
    cur[0] = 0; cur[1] = 0;
  }
}
// Block -> rank placement on the device (partitioning/LPTScheduler.scala:57-76: longest processing time first, cost
// of a block = records x entities), re-evaluated from the GLOBAL block sizes of the state just produced, so every
// rank computes the same table.  The new table only re-routes: blocks migrate with the next exchange as ordinary
// cluster messages.  Adopted only when the current table is more than `threshold` above the LPT makespan.
__global__ void k_lpt(int P, int world, int ent_slot, int rec_slot, const long long *__restrict__ glob,
                      long long *__restrict__ ctl, int period, double threshold, int *__restrict__ owner,
                      int *__restrict__ scratch /* 2*P ints */, double *__restrict__ dscratch /* P + world doubles */) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  if (sweep_dead(ctl) || period <= 0 || ((ctl[CTL_ITER] + 1) % period) != 0) return;
  int *order = scratch, *cand = scratch + P;
  double *cost = dscratch, *load = dscratch + P;
  double total = 0.0;
  for (int b = 0; b < P; ++b) {
    cost[b] = (double)glob[ent_slot + b] * (double)glob[rec_slot + b];
    total += cost[b];
    order[b] = b;
  }
  if (!(total > 0.0)) return;
  for (int i = 1; i < P; ++i) {  // insertion sort by (-cost, block id)
    const int b = order[i];
    int j = i - 1;
    while (j >= 0 && (cost[order[j]] < cost[b] || (cost[order[j]] == cost[b] && order[j] > b))) { order[j + 1] = order[j]; --j; }
    order[j + 1] = b;
  }
  for (int r = 0; r < world; ++r) load[r] = 0.0;
  for (int i = 0; i < P; ++i) {
    const int b = order[i];
    int best = 0;
    for (int r = 1; r < world; ++r) if (load[r] < load[best]) best = r;
    cand[b] = best;
    load[best] += cost[b];
  }
  double lpt_max = 0.0;
  for (int r = 0; r < world; ++r) lpt_max = fmax(lpt_max, load[r]);
  for (int r = 0; r < world; ++r) load[r] = 0.0;
  for (int b = 0; b < P; ++b) load[owner[b]] += cost[b];
  double cur_max = 0.0;
  for (int r = 0; r < world; ++r) cur_max = fmax(cur_max, load[r]);
  if (cur_max > threshold * lpt_max) {
    for (int b = 0; b < P; ++b) owner[b] = cand[b];
    ctl[CTL_REPLACED] += 1;
  }
}

// ---- (2) host-mediated exchange (multi-node / no peer access): counts to the host, messages packed into caller
// buffers, the host moves them (e.g. NCCL all-to-all) and hands back what arrived -----------------------------------
__global__ void k_move_count_ent(int64_t E, const int *__restrict__ blk, const int *__restrict__ owner, int rank,
                                 const unsigned char *__restrict__ ent_owned, int *__restrict__ ent_dest,
                                 unsigned long long *__restrict__ cnt) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= E) return;
  int d = -1;
  if (ent_owned[e]) {
    const int o = owner[blk[e]];
    if (o != rank) { d = o; atomicAdd(&cnt[o], 1ull); }
  }
  ent_dest[e] = d;
}
__global__ void k_move_count_rec(int64_t R, const int *__restrict__ link, const unsigned char *__restrict__ rec_owned,
                                 const int *__restrict__ ent_dest, unsigned long long *__restrict__ cnt) {
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= R || !rec_owned[r]) return;
  const int d = ent_dest[link[r]];
  if (d >= 0) atomicAdd(&cnt[d], 1ull);
}
__global__ void k_move_pack_ent(int64_t E, int A, const int *__restrict__ y, const int *__restrict__ ent_dest,
                                unsigned char *__restrict__ ent_owned, unsigned long long *__restrict__ cursor,
                                int *__restrict__ buf) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= E) return;
  const int d = ent_owned[e] ? ent_dest[e] : -1;
  if (d < 0) return;
  const unsigned long long slot = atomicAdd(&cursor[d], 1ull);
  int *m = buf + slot * (A + 1);
  m[0] = (int)e;
  for (int a = 0; a < A; ++a) m[1 + a] = y[e * A + a];
  ent_owned[e] = 0;
}
__global__ void k_move_pack_rec(int64_t R, const int *__restrict__ link, const unsigned *__restrict__ zmask,
                                const int *__restrict__ ent_dest, unsigned char *__restrict__ rec_owned,
                                unsigned long long *__restrict__ cursor, int *__restrict__ buf) {
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= R || !rec_owned[r]) return;
  const int d = ent_dest[link[r]];
  if (d < 0) return;
  const unsigned long long slot = atomicAdd(&cursor[d], 1ull);
  int *m = buf + slot * 3;
  m[0] = (int)r; m[1] = link[r]; m[2] = (int)zmask[r];
  rec_owned[r] = 0;
}
__global__ void k_unpack_ent(int64_t n, int A, const int *__restrict__ buf, const AttrDev *__restrict__ attrs,
                             TreeDev tree, int *__restrict__ y, double *__restrict__ entN, int *__restrict__ blk,
                             unsigned char *__restrict__ ent_owned) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int *m = buf + i * (A + 1);
  const int64_t e = m[0];
  double nn = 1.0;
  for (int a = 0; a < A; ++a) {
    const int v = m[1 + a];
    y[e * A + a] = v;
    if (!attrs[a].is_const) nn = nn * attrs[a].norm[v];
  }
  entN[e] = nn;
  blk[e] = tree.n_nodes > 0 ? tree_leaf(tree, m + 1) : 0;
  ent_owned[e] = 1;
}
__global__ void k_unpack_rec(int64_t n, const int *__restrict__ buf, int *__restrict__ link,
                             unsigned *__restrict__ zmask, unsigned char *__restrict__ rec_owned) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int *m = buf + i * 3;
  const int64_t r = m[0];
  link[r] = m[1];
  zmask[r] = (unsigned)m[2];
  rec_owned[r] = 1;
}

// ---- read-out of a sharded state --------------------------------------------------------------------------
// owned rows of the state into caller-provided device buffers, zeros elsewhere (summing over ranks = full state)
__global__ void k_export_ent(int64_t E, int A, const unsigned char *__restrict__ owned, const int *__restrict__ y,
                             const int *__restrict__ blk, int *__restrict__ y_out, int *__restrict__ blk_out) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= E) return;
  const bool o = owned[e];
  for (int a = 0; a < A; ++a) y_out[e * A + a] = o ? y[e * A + a] : 0;
  blk_out[e] = o ? blk[e] : 0;
}
__global__ void k_export_rec(int64_t R, int A, const unsigned char *__restrict__ owned, const int *__restrict__ link,
                             const unsigned *__restrict__ zmask, int *__restrict__ link_out,
                             unsigned char *__restrict__ z_out) {
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= R) return;
  const bool o = owned[r];
  link_out[r] = o ? link[r] : 0;
  const unsigned zm = o ? zmask[r] : 0u;
  for (int a = 0; a < A; ++a) z_out[r * A + a] = (zm >> a) & 1u;
}
// owned rows only, compacted in the order of ent_sorted / rec_sorted (block-major): ids + rows
__global__ void k_gather_ent(int64_t n, int A, const int *__restrict__ ent_sorted, const int *__restrict__ y,
                             const int *__restrict__ blk, int *__restrict__ ids, int *__restrict__ y_out,
                             int *__restrict__ blk_out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int64_t e = ent_sorted[i];
  ids[i] = (int)e;
  for (int a = 0; a < A; ++a) y_out[i * A + a] = y[e * A + a];
  blk_out[i] = blk[e];
}
__global__ void k_gather_rec(int64_t n, int A, const int *__restrict__ rec_sorted, const int *__restrict__ link,
                             const unsigned *__restrict__ zmask, int *__restrict__ ids, int *__restrict__ link_out,
                             unsigned char *__restrict__ z_out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int64_t r = rec_sorted[i];
  ids[i] = (int)r;
  link_out[i] = link[r];
  const unsigned zm = zmask[r];
  for (int a = 0; a < A; ++a) z_out[i * A + a] = (zm >> a) & 1u;
}
// Order-independent 64-bit fingerprint of the owned rows: sum over rows of a mixed hash of (row id, row contents).
// Sums of the per-rank values (mod 2^64) are the same for every rank count and placement.
__device__ __forceinline__ unsigned long long mix64(unsigned long long z) {
  z += 0x9E3779B97F4A7C15ull;
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  return z ^ (z >> 31);
}
__global__ void __launch_bounds__(256) k_state_hash(RowSet ents, RowSet recs, int A, const int *__restrict__ y,
                                                    const int *__restrict__ link, const unsigned *__restrict__ zmask,
                                                    unsigned long long *__restrict__ out /*2*/) {
  unsigned long long he = 0, hr = 0;
  const int64_t ne = ents.count(), nr = recs.count();
  GRID_STRIDE(i, ne) {
    const int64_t e = ents.row(i);
    if (e < 0) continue;
    unsigned long long h = mix64(0xE000000000000000ull ^ (unsigned long long)e);
    for (int a = 0; a < A; ++a) h = mix64(h ^ (unsigned long long)(unsigned)y[e * A + a]);
    he += h;
  }
  GRID_STRIDE(i, nr) {
    const int64_t r = recs.row(i);
    if (r < 0) continue;
    unsigned long long h = mix64(0xA000000000000000ull ^ (unsigned long long)r);
    h = mix64(h ^ (unsigned long long)(unsigned)link[r]);
    h = mix64(h ^ (unsigned long long)zmask[r]);
    hr += h;
  }
  typedef cub::BlockReduce<unsigned long long, 256> BR;
  __shared__ typename BR::TempStorage t1, t2;
  const unsigned long long se = BR(t1).Sum(he), sr = BR(t2).Sum(hr);
  if (threadIdx.x == 0) { atomicAdd(&out[0], se); atomicAdd(&out[1], sr); }
}

// ---------------------------------------------------------------------------------------------------
// host-side context
// ---------------------------------------------------------------------------------------------------
template <typename T>
struct DevBuf {
  T *p = nullptr;
  size_t n = 0;
  cudaError_t alloc(size_t count) {
    release();
    n = count;
    return cudaMalloc((void **)&p, std::max<size_t>(count, 1) * sizeof(T));
  }
  void release() { if (p) cudaFree(p); p = nullptr; n = 0; }
  ~DevBuf() { release(); }
};

// what dbl_comm_export hands to the peers (DBL_COMM_BLOB_BYTES)
struct CommBlob {
  uint32_t magic;
  int32_t rank, world, device;
  int64_t pid;
  uint64_t ptr;  // address in the exporting process (used when the importer IS that process)
  uint64_t bytes;
  int64_t E, R;
  int32_t A, nws;
  cudaIpcMemHandle_t handle;
  char pad[DBL_COMM_BLOB_BYTES - 4 - 12 - 8 - 8 - 8 - 16 - 8 - (int)sizeof(cudaIpcMemHandle_t)];
};
static_assert(sizeof(CommBlob) == DBL_COMM_BLOB_BYTES, "blob layout");
constexpr uint32_t COMM_MAGIC = 0xDB1B2002u;

struct dbl_ctx {
  int A = 0, F = 0, P = 1, device = 0;
  uint64_t seed = 0;
  int rank = 0, world = 1;
  std::vector<double> alpha, beta;
  std::string err;
  cudaStream_t stream = nullptr;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;

  // model (device)
  std::vector<DevBuf<double>> dtab;  // per-attr double tables
  std::vector<DevBuf<int>> itab;
  DevBuf<AttrDev> attrs;
  DevBuf<int> perm_dev;
  int perm[DBL_MAX_ATTRS] = {0};
  int n_str = 0;       // non-constant attributes
  int pack_consts = 0; // constant attributes byte-packed into the tiles (0 = none)
  int hslots = 32, hshift = 27;  // common hash-table size of the non-constant attributes; hslots = 0: none
  std::vector<AttrDev> h_attrs;
  DevBuf<int> tree_buf;
  TreeDev tree{};
  DevBuf<double> prior;  // alpha[A], beta[A], file sizes[F] (k_theta)

  // state
  int64_t R = 0, E = 0, iteration = 0;
  bool has_state = false;
  DevBuf<int> x, file, link, newlink, y, blk;
  DevBuf<uint8_t> zbytes;  // staging for the byte-per-flag host format of z
  DevBuf<int> vflag, file_cnt;
  DevBuf<unsigned> zmask;
  DevBuf<double> entN;
  std::vector<double> h_theta, h_file_sizes_d;
  std::vector<int64_t> file_sizes;
  long long h_head[2] = {0, 0};  // staging of (iteration, status) for a new state

  // control block (one allocation, mirrored in pinned host memory by snapshot()):
  //   [CTL_WORDS] ctl | [nw] partial summary | [nw] global summary | [A*F] theta | [A*F] theta_prev | [2] hash
  DevBuf<long long> cb;
  long long *h_cb = nullptr;  // pinned
  size_t cb_words = 0;
  int nw = 0;  // summary words: A*F + (A+1) + 2 + 2*P
  long long *ctl() const { return cb.p; }
  unsigned long long *part() const { return reinterpret_cast<unsigned long long *>(cb.p + CTL_WORDS); }
  long long *glob() const { return cb.p + CTL_WORDS + nw; }
  double *theta() const { return reinterpret_cast<double *>(cb.p + CTL_WORDS + 2 * (size_t)nw); }
  double *theta_prev() const { return theta() + (size_t)A * F; }
  unsigned long long *hash_words() const { return reinterpret_cast<unsigned long long *>(theta_prev() + (size_t)A * F); }
  const long long *h_ctl() const { return h_cb; }
  const long long *h_part() const { return h_cb + CTL_WORDS; }
  const long long *h_glob() const { return h_cb + CTL_WORDS + nw; }
  const double *h_theta_dev() const { return reinterpret_cast<const double *>(h_cb + CTL_WORDS + 2 * (size_t)nw); }
  int n_counts() const { return A * F + (A + 1) + 2; }  // words a host-mediated all-reduce carries
  int iso_slot() const { return A * F + (A + 1); }
  int ll_slot() const { return A * F + (A + 1) + 1; }
  int blk_ent_slot() const { return n_counts(); }
  int blk_rec_slot() const { return n_counts() + P; }

  // ownership (multi-GPU sharding by block)
  std::vector<int> owner_h;  // P entries; default: everything owned by this rank
  DevBuf<int> owner, ent_dest, ent_key, link_key;
  DevBuf<unsigned char> ent_owned, rec_owned;
  DevBuf<unsigned long long> move_cnt;  // host-mediated exchange: [2*world] counts then [2*world] cursors
  std::vector<int64_t> h_move_ent, h_move_rec;
  bool in_sweep = false, in_block_sweep = false;
  int block_sampler = 0;
  std::vector<char> block_done;
  DevBuf<int> blk_frozen;
  bool all_owned = true;  // no shard has been carved out of the replicated state yet

  // peer-to-peer exchange
  DevBuf<unsigned char> comm_buf;
  size_t comm_bytes = 0;
  CommDev comm{};
  bool comm_ready = false;
  std::vector<void *> ipc_opened;
  DevBuf<int> lpt_scratch;
  DevBuf<double> lpt_dscratch;
  int rebalance_period = 16;
  double rebalance_threshold = 1.03;
  long long barrier_timeout_cycles = 120000000000LL;  // ~60 s at 1.9 GHz: ranks may reach their first sweep far apart

  // layout
  DevBuf<int> iota, blk_sorted, ent_sorted, rec_key, rec_key_sorted, rec_sorted;
  DevBuf<int> ent_ptr, tile_ptr, rec_ptr, cta_ptr, cta_ptr2, cta_ptr3, tiles, qtiles;
  DevBuf<double> lane_sums;  // k_link_pcg2 scratch: pass-1 lane sums per chunk of every resident warp
  int qtile_pk = 0;  // quad tiles carry the packed constants (PK instantiations of k_link_pcg2)
  bool tiles_valid[2] = {false, false};  // attribute-major / quad tiles match the current layout
  // inverted index of the block tables for the pruned PCG-I link kernel (built on demand, once per sweep)
  DevBuf<unsigned long long> inv_key_in, inv_key;
  DevBuf<unsigned> inv_key32_in, inv_key32;
  DevBuf<int> inv_pos_in, inv_pos, inv_seg, inv_vptr, heavy_list;
  InvDense inv_dense;
  bool inv_use_dense = false;
  DevBuf<unsigned char> inv_tmp;
  size_t inv_tmp_bytes = 0;
  bool inv_valid = false;
  int inv_vbits = 32;
  DevBuf<int> link_sorted, rec_by_ent, ent_rec_ptr;
  DevBuf<unsigned char> rec_class;  // static cost class of a record (k_rec_class)
  DevBuf<unsigned char> cub_tmp;
  size_t cub_bytes = 0;
  int max_ctas = 0;
  DevBuf<int> gather_i;  // staging of dbl_download_owned
  DevBuf<unsigned char> gather_b;

  // host copies refreshed by snapshot()
  int64_t h_pairs = 0;
  int64_t h_owned_ent = -1, h_owned_rec = -1;  // -1 = not known on the host since the last re-partitioning

  int64_t launches = 0;
  double link_ms = 0.0;
  int link_mode = 0;  // 0 auto, 1 generic kernel everywhere, 2 dense TMA kernels everywhere (no pruning)
  double last_sweep_ms = 0.0;
  int64_t link_launches = 0;
  // eager sweeps are timed phase by phase: events before / after the link kernel, after the value / distortion /
  // summary kernels, after the exchange, after the re-layout
  struct PhaseEvents { cudaEvent_t e[5]; };
  std::vector<PhaseEvents> pending_events, event_pool;
  PhaseEvents cur_events{};
  bool cur_timed = false;
  double phase_ms[4] = {0, 0, 0, 0};
  int64_t phase_sweeps = 0;
  size_t pcg2_smem_cfg = 0, match_smem_cfg = 0;  // dynamic shared memory opted in on THIS device
  int sm_count = 148;
  int pcg2_grid = 148 * DBL_PCG2_CTAS_PER_SM;   // persistent CTAs of k_link_pcg2
  int pcg2_recs = LINK_WARPS;                   // records per work item of k_link_pcg2
  bool async_open = false;  // sweeps enqueued by dbl_sweep_async, not yet collected by dbl_sync
  // CUDA graphs of one sweep (launch-bound problem sizes): key = sampler * 4 + link mode
  struct SweepGraph { cudaGraph_t graph = nullptr; cudaGraphExec_t exec = nullptr; int64_t launches = 0; };
  std::map<int, SweepGraph> graphs;
  std::map<int, bool> graph_warm;  // one eager sweep of that kind has run (lazy allocations, shared-memory opt-ins)
  int graph_mode = 0;              // 0 auto (small problems), 1 never, 2 always
  bool capturing = false;
  void drop_graphs() {
    for (auto &kv : graphs) {
      if (kv.second.exec) cudaGraphExecDestroy(kv.second.exec);
      if (kv.second.graph) cudaGraphDestroy(kv.second.graph);
    }
    graphs.clear();
    graph_warm.clear();
  }

  void set_error(const std::string &s) { err = s; }
};

static inline int grid_for(int64_t n, int bs) { return (int)std::max<int64_t>(1, (n + bs - 1) / bs); }
// grid of a grid-stride kernel over at most n rows
static inline int grid_rows(int64_t n, int bs) {
  return (int)std::min<int64_t>(148 * (2048 / bs), std::max<int64_t>(1, (n + bs - 1) / bs));
}

static RowSet rows_prefix(dbl_ctx *ctx, bool ents) {
  RowSet r;
  r.ctl = ctx->ctl();
  r.sorted = ents ? ctx->ent_sorted.p : ctx->rec_sorted.p;
  r.owned = nullptr;
  r.n_all = ents ? ctx->E : ctx->R;
  r.count_word = ents ? CTL_OWNED_ENT : CTL_OWNED_REC;
  return r;
}
static RowSet rows_masked(dbl_ctx *ctx, bool ents) {
  RowSet r;
  r.ctl = ctx->ctl();
  r.sorted = nullptr;
  r.owned = ents ? ctx->ent_owned.p : ctx->rec_owned.p;
  r.n_all = ents ? ctx->E : ctx->R;
  r.count_word = ents ? CTL_OWNED_ENT : CTL_OWNED_REC;
  return r;
}

static int upload_tree(dbl_ctx *ctx, const dbl_kdtree *t) {
  if (t) {
    const int n = t->n_nodes;
    std::vector<int> pack;
    pack.insert(pack.end(), t->attr.begin(), t->attr.end());
    pack.insert(pack.end(), t->kind.begin(), t->kind.end());
    pack.insert(pack.end(), t->split.begin(), t->split.end());
    pack.insert(pack.end(), t->set_ptr.begin(), t->set_ptr.end());
    pack.insert(pack.end(), t->leaf_no.begin(), t->leaf_no.end());
    pack.insert(pack.end(), t->set_val.begin(), t->set_val.end());
    for (int i = 0; i < n; ++i)
      if (t->attr[i] >= ctx->A) { ctx->set_error("partitioner attribute id out of range"); return DBL_ERR_INVALID; }
    CUDA_TRY(ctx->tree_buf.alloc(pack.size()));
    CUDA_TRY(cudaMemcpy(ctx->tree_buf.p, pack.data(), pack.size() * sizeof(int), cudaMemcpyHostToDevice));
    int *base = ctx->tree_buf.p;
    ctx->tree.n_nodes = n;
    ctx->tree.attr = base;
    ctx->tree.kind = base + n;
    ctx->tree.split = base + 2 * n;
    ctx->tree.set_ptr = base + 3 * n;
    ctx->tree.leaf_no = base + 3 * n + (n + 1);
    ctx->tree.set_val = base + 4 * n + (n + 1);
    ctx->P = t->n_leaves;
  } else {
    ctx->tree.n_nodes = 0;
    ctx->P = 1;
  }
  return DBL_OK;
}

static int upload_model(dbl_ctx *ctx, const dbl_model_desc *d) {
  const int A = d->num_attrs;
  ctx->h_attrs.resize(A);
  ctx->dtab.resize((size_t)A * 11);
  ctx->itab.resize((size_t)A * 4);
  auto up_d = [&](DevBuf<double> &b, const std::vector<double> &v) -> cudaError_t {
    cudaError_t e = b.alloc(v.size());
    if (e != cudaSuccess) return e;
    if (v.empty()) return cudaSuccess;
    return cudaMemcpy(b.p, v.data(), v.size() * sizeof(double), cudaMemcpyHostToDevice);
  };
  auto up_i = [&](DevBuf<int> &b, const std::vector<int32_t> &v) -> cudaError_t {
    cudaError_t e = b.alloc(v.size());
    if (e != cudaSuccess) return e;
    if (v.empty()) return cudaSuccess;
    return cudaMemcpy(b.p, v.data(), v.size() * sizeof(int), cudaMemcpyHostToDevice);
  };
  // one hash-table size for the whole model: re-hash the smaller tables to the largest
  int Hmax = 32;
  bool hash_ok = true;
  for (int a = 0; a < A; ++a) {
    if (d->indexes[a]->is_const) continue;
    if (d->indexes[a]->hsize <= 0) hash_ok = false;
    Hmax = std::max(Hmax, d->indexes[a]->hsize);
  }
  std::vector<dbl_index> rehashed(A);
  for (int a = 0; a < A; ++a) {
    const dbl_index *ix = d->indexes[a];
    if (hash_ok && !ix->is_const && ix->hsize != Hmax) {
      rehashed[a] = *ix;
      rehashed[a].build_hash(Hmax);
      if (rehashed[a].hsize != Hmax) hash_ok = false;
      ix = &rehashed[a];
    }
    DevBuf<double> *t = &ctx->dtab[(size_t)a * 11];
    DevBuf<int> *ti = &ctx->itab[(size_t)a * 4];
    CUDA_TRY(up_d(t[0], ix->phi));
    CUDA_TRY(up_d(t[1], ix->probs));
    CUDA_TRY(up_d(t[2], ix->norm));
    CUDA_TRY(up_d(t[3], ix->invnorm));
    CUDA_TRY(up_d(t[4], ix->pk));
    CUDA_TRY(up_d(t[5], ix->cdf));
    CUDA_TRY(up_d(t[6], ix->logphi));
    CUDA_TRY(up_d(t[7], ix->lognorm));
    CUDA_TRY(up_d(t[8], ix->expsim));
    CUDA_TRY(up_i(ti[0], ix->rowptr));
    CUDA_TRY(up_i(ti[1], ix->col));
    CUDA_TRY(up_d(t[9], ix->hvals));
    {
      std::vector<double> diag(ix->V, 1.0);  // E(v, v) (AttributeIndex.expSimOf(v, v)); 1 when the row has no entry
      for (int v = 0; v < ix->V && !ix->is_const; ++v)
        for (int q = ix->rowptr[v]; q < ix->rowptr[v + 1]; ++q)
          if (ix->col[q] == v) diag[v] = ix->expsim[q];
      CUDA_TRY(up_d(t[10], diag));
    }
    CUDA_TRY(up_i(ti[2], ix->hkeys));
    {
      std::vector<int32_t> hm(ix->hmult.begin(), ix->hmult.end());
      CUDA_TRY(up_i(ti[3], hm));
    }
    AttrDev &h = ctx->h_attrs[a];
    h.V = ix->V; h.is_const = ix->is_const ? 1 : 0; h.kmax = ix->kmax; h.hsize = ix->hsize;
    h.hshift = ix->hshift; h.pad0 = h.pad1 = h.pad2 = 0;
    h.hvals = t[9].p; h.hkeys = ti[2].p; h.hmult = reinterpret_cast<const unsigned *>(ti[3].p);
    h.phi = t[0].p; h.probs = t[1].p; h.norm = t[2].p; h.invnorm = t[3].p; h.pk = t[4].p; h.cdf = t[5].p;
    h.logphi = t[6].p; h.lognorm = t[7].p; h.expsim = t[8].p; h.diag = t[10].p;
    h.rowptr = ti[0].p; h.col = ti[1].p;
  }
  CUDA_TRY(ctx->attrs.alloc(A));
  CUDA_TRY(cudaMemcpy(ctx->attrs.p, ctx->h_attrs.data(), sizeof(AttrDev) * A, cudaMemcpyHostToDevice));
  {
    int k = 0;
    for (int a = 0; a < A; ++a) if (ctx->h_attrs[a].is_const) ctx->perm[k++] = a;
    ctx->n_str = A - k;
    // byte-packed copy of the constant attributes in the tiles (k_link_pcg2): 1..4 of them, every vocabulary <= 255
    ctx->pack_consts = (k >= 1 && k <= 4) ? k : 0;
    for (int q = 0; q < k; ++q) if (ctx->h_attrs[ctx->perm[q]].V > 255) ctx->pack_consts = 0;
    if (getenv("DBL_NO_PACK")) ctx->pack_consts = 0;  // tests: the unpacked kernels on a packable model
    for (int a = 0; a < A; ++a) if (!ctx->h_attrs[a].is_const) ctx->perm[k++] = a;
    ctx->hslots = hash_ok ? Hmax : 0;
    ctx->hshift = 32;
    for (int h2 = 1; h2 < Hmax; h2 <<= 1) ctx->hshift -= 1;
    CUDA_TRY(ctx->perm_dev.alloc(A));
    CUDA_TRY(cudaMemcpy(ctx->perm_dev.p, ctx->perm, sizeof(int) * A, cudaMemcpyHostToDevice));
  }
  return upload_tree(ctx, d->tree);
}

// (re)allocate the control block for the current number of blocks; the global summary and theta survive
static int alloc_control(dbl_ctx *ctx) {
  const int A = ctx->A, F = ctx->F;
  const int nw = ctx->n_counts() + 2 * ctx->P;
  const size_t words = CTL_WORDS + 2 * (size_t)nw + 2 * (size_t)A * F + 2;
  if (ctx->cb.p && ctx->nw == nw) return DBL_OK;
  std::vector<long long> keep_ctl(CTL_WORDS, 0), keep_glob(ctx->n_counts(), 0);
  std::vector<double> keep_theta(2 * (size_t)A * F, 0.0);
  const bool had = ctx->cb.p != nullptr;
  if (had) {
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    CUDA_TRY(cudaMemcpy(keep_ctl.data(), ctx->ctl(), sizeof(long long) * CTL_WORDS, cudaMemcpyDeviceToHost));
    CUDA_TRY(cudaMemcpy(keep_glob.data(), ctx->glob(), sizeof(long long) * ctx->n_counts(), cudaMemcpyDeviceToHost));
    CUDA_TRY(cudaMemcpy(keep_theta.data(), ctx->theta(), sizeof(double) * 2 * A * F, cudaMemcpyDeviceToHost));
  }
  CUDA_TRY(ctx->cb.alloc(words));
  ctx->cb_words = words;
  ctx->nw = nw;
  if (ctx->h_cb) cudaFreeHost(ctx->h_cb);
  CUDA_TRY(cudaMallocHost((void **)&ctx->h_cb, words * sizeof(long long)));
  memset(ctx->h_cb, 0, words * sizeof(long long));
  CUDA_TRY(cudaMemset(ctx->cb.p, 0, words * sizeof(long long)));
  if (had) {
    CUDA_TRY(cudaMemcpy(ctx->ctl(), keep_ctl.data(), sizeof(long long) * CTL_WORDS, cudaMemcpyHostToDevice));
    CUDA_TRY(cudaMemcpy(ctx->glob(), keep_glob.data(), sizeof(long long) * ctx->n_counts(), cudaMemcpyHostToDevice));
    CUDA_TRY(cudaMemcpy(ctx->theta(), keep_theta.data(), sizeof(double) * 2 * A * F, cudaMemcpyHostToDevice));
  }
  return DBL_OK;
}

// for hosts without CUDA bindings of their own (a JVM through JNI): the device of the contexts this thread creates
extern "C" int dbl_set_device(int32_t device) { return cudaSetDevice(device) == cudaSuccess ? DBL_OK : DBL_ERR_CUDA; }
extern "C" int32_t dbl_device_count(void) {
  int n = 0;
  return cudaGetDeviceCount(&n) == cudaSuccess ? n : 0;
}

extern "C" int dbl_ctx_create(dbl_ctx **out, const dbl_model_desc *d) {
  if (!out || !d || d->num_attrs <= 0 || d->num_attrs > DBL_MAX_ATTRS || d->num_files <= 0 || !d->indexes ||
      !d->alpha || !d->beta)
    return DBL_ERR_INVALID;
  for (int a = 0; a < d->num_attrs; ++a)
    if (!d->indexes[a] || !(d->alpha[a] > 0.0) || !(d->beta[a] > 0.0)) return DBL_ERR_INVALID;  // package.scala:165
  if (d->world_size > MAX_WORLD || d->rank < 0 || (d->world_size > 0 && d->rank >= d->world_size)) return DBL_ERR_INVALID;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return DBL_ERR_CUDA;  // no CPU fallback
  auto *ctx = new dbl_ctx();
  ctx->A = d->num_attrs;
  ctx->F = d->num_files;
  ctx->seed = d->seed;
  ctx->rank = d->rank;
  ctx->world = d->world_size > 0 ? d->world_size : 1;
  ctx->alpha.assign(d->alpha, d->alpha + ctx->A);
  ctx->beta.assign(d->beta, d->beta + ctx->A);
  cudaGetDevice(&ctx->device);
  {
    int sms = 0;
    if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, ctx->device) == cudaSuccess && sms > 0)
      ctx->sm_count = sms;
  }
  *out = ctx;
  CUDA_TRY(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
  CUDA_TRY(cudaEventCreate(&ctx->ev0));
  CUDA_TRY(cudaEventCreate(&ctx->ev1));
  int rc = upload_model(ctx, d);
  if (rc != DBL_OK) return rc;
  rc = alloc_control(ctx);
  if (rc != DBL_OK) return rc;
  CUDA_TRY(ctx->prior.alloc(2 * (size_t)ctx->A + ctx->F));
  {
    std::vector<double> pr(2 * (size_t)ctx->A + ctx->F, 0.0);
    std::copy(ctx->alpha.begin(), ctx->alpha.end(), pr.begin());
    std::copy(ctx->beta.begin(), ctx->beta.end(), pr.begin() + ctx->A);
    CUDA_TRY(cudaMemcpy(ctx->prior.p, pr.data(), pr.size() * sizeof(double), cudaMemcpyHostToDevice));
  }
  ctx->h_theta.assign((size_t)ctx->A * ctx->F, 0.0);
  return DBL_OK;
}

static void comm_close(dbl_ctx *ctx) {
  for (void *p : ctx->ipc_opened) cudaIpcCloseMemHandle(p);
  ctx->ipc_opened.clear();
  ctx->comm_ready = false;
}

extern "C" void dbl_ctx_destroy(dbl_ctx *ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  if (ctx->stream) cudaStreamSynchronize(ctx->stream);
  comm_close(ctx);
  ctx->drop_graphs();
  for (auto &pe : ctx->pending_events) for (cudaEvent_t e : pe.e) cudaEventDestroy(e);
  for (auto &pe : ctx->event_pool) for (cudaEvent_t e : pe.e) cudaEventDestroy(e);
  if (ctx->ev0) cudaEventDestroy(ctx->ev0);
  if (ctx->ev1) cudaEventDestroy(ctx->ev1);
  if (ctx->stream) cudaStreamDestroy(ctx->stream);
  if (ctx->h_cb) cudaFreeHost(ctx->h_cb);
  delete ctx;
}
extern "C" const char *dbl_last_error(const dbl_ctx *ctx) { return ctx ? ctx->err.c_str() : "null context"; }
extern "C" int64_t dbl_num_records(const dbl_ctx *ctx) { return ctx ? ctx->R : 0; }
extern "C" int64_t dbl_num_entities(const dbl_ctx *ctx) { return ctx ? ctx->E : 0; }
extern "C" int64_t dbl_iteration(const dbl_ctx *ctx) { return ctx ? ctx->iteration : 0; }
extern "C" int64_t dbl_kernel_launches(const dbl_ctx *ctx) { return ctx ? ctx->launches : 0; }
extern "C" const char *dbl_version(void) { return "dblink_b200 0.2 (sm_100a)"; }

static int alloc_blocks(dbl_ctx *ctx) {
  const int P = ctx->P;
  ctx->drop_graphs();  // captured sweeps hold the old buffers / tree
  if ((int)ctx->owner_h.size() != P) ctx->owner_h.assign(P, ctx->rank);
  CUDA_TRY(ctx->owner.alloc(P));
  CUDA_TRY(cudaMemcpy(ctx->owner.p, ctx->owner_h.data(), sizeof(int) * P, cudaMemcpyHostToDevice));
  CUDA_TRY(ctx->ent_ptr.alloc(P + 1));
  CUDA_TRY(ctx->tile_ptr.alloc(P + 1));
  CUDA_TRY(ctx->rec_ptr.alloc(P + 1));
  CUDA_TRY(ctx->cta_ptr.alloc(P + 1));
  CUDA_TRY(ctx->cta_ptr2.alloc(P + 1));
  CUDA_TRY(ctx->cta_ptr3.alloc(P + 1));
  CUDA_TRY(ctx->lpt_scratch.alloc(2 * (size_t)P));
  CUDA_TRY(ctx->lpt_dscratch.alloc((size_t)P + MAX_WORLD));
  const size_t max_tiles = (size_t)(ctx->E / TE) + (size_t)P + 1;
  CUDA_TRY(ctx->tiles.alloc(max_tiles * tile_words(ctx->A)));
  ctx->qtile_pk = (ctx->pack_consts && ctx->hslots == 32) ? 1 : 0;
  {
    // work item and grid of the persistent PCG-II kernel for this model shape (see pcg2_rpw)
    const int hc = ctx->hslots == 32 ? 32 : 0;
    ctx->pcg2_recs = pcg2_warps(hc, ctx->n_str) * pcg2_rpw(hc, ctx->n_str);
    ctx->pcg2_grid = ctx->sm_count * pcg2_ctas_per_sm(hc, ctx->n_str);
    const size_t need = (size_t)ctx->pcg2_grid * ctx->pcg2_recs * 1024;
    if (ctx->lane_sums.n < need) CUDA_TRY(ctx->lane_sums.alloc(need));
  }
  CUDA_TRY(ctx->qtiles.alloc(max_tiles * qtile_words(qtile_nv(ctx->A, ctx->n_str, ctx->qtile_pk != 0)) * TE));
  ctx->max_ctas = (int)((ctx->R + LINK_WARPS - 1) / LINK_WARPS) + P;
  return alloc_control(ctx);
}

static int alloc_state(dbl_ctx *ctx, int64_t R, int64_t E) {
  const int A = ctx->A;
  if (R <= 0 || E <= 0 || R > 0x7fffffff || E > 0x7fffffff) { ctx->set_error("bad R/E"); return DBL_ERR_INVALID; }
  ctx->all_owned = true;
  if (ctx->R == R && ctx->E == E && ctx->x.p && ctx->tiles.p) {  // same shape as the previous state: reuse buffers
    CUDA_TRY(cudaMemsetAsync(ctx->ent_owned.p, 1, E, ctx->stream));
    CUDA_TRY(cudaMemsetAsync(ctx->rec_owned.p, 1, R, ctx->stream));
    return DBL_OK;
  }
  if (ctx->comm_ready || ctx->comm_buf.p) {  // the communication buffers were sized for the old state
    comm_close(ctx);
    ctx->comm_buf.release();
  }
  ctx->R = R; ctx->E = E;
  ctx->drop_graphs();
  CUDA_TRY(ctx->zbytes.alloc((size_t)R * A));
  CUDA_TRY(ctx->vflag.alloc(1));
  CUDA_TRY(ctx->file_cnt.alloc(ctx->F));
  CUDA_TRY(ctx->x.alloc((size_t)R * A));
  CUDA_TRY(ctx->file.alloc(R));
  CUDA_TRY(ctx->link.alloc(R));
  CUDA_TRY(ctx->newlink.alloc(R));
  CUDA_TRY(ctx->zmask.alloc(R));
  CUDA_TRY(ctx->y.alloc((size_t)E * A));
  CUDA_TRY(ctx->blk.alloc(E));
  CUDA_TRY(ctx->entN.alloc(E));
  CUDA_TRY(ctx->ent_owned.alloc(E));
  CUDA_TRY(ctx->rec_owned.alloc(R));
  CUDA_TRY(ctx->rec_class.alloc(R));
  CUDA_TRY(cudaMemsetAsync(ctx->ent_owned.p, 1, E, ctx->stream));
  CUDA_TRY(cudaMemsetAsync(ctx->rec_owned.p, 1, R, ctx->stream));
  CUDA_TRY(ctx->ent_dest.alloc(E));
  CUDA_TRY(ctx->ent_key.alloc(E));
  CUDA_TRY(ctx->link_key.alloc(R));
  CUDA_TRY(ctx->move_cnt.alloc(4 * (size_t)ctx->world));
  const int64_t M = std::max(R, E);
  CUDA_TRY(ctx->iota.alloc(M));
  k_iota<<<grid_for(M, 256), 256, 0, ctx->stream>>>(M, ctx->iota.p);
  CUDA_TRY(ctx->blk_sorted.alloc(E));
  CUDA_TRY(ctx->ent_sorted.alloc(E));
  CUDA_TRY(ctx->rec_key.alloc(R));
  CUDA_TRY(ctx->rec_key_sorted.alloc(R));
  CUDA_TRY(ctx->rec_sorted.alloc(R));
  { int rc = alloc_blocks(ctx); if (rc) return rc; }
  CUDA_TRY(ctx->link_sorted.alloc(R));
  CUDA_TRY(ctx->rec_by_ent.alloc(R));
  CUDA_TRY(ctx->ent_rec_ptr.alloc(E + 1));
  size_t b1 = 0, b2 = 0;
  cub::DeviceRadixSort::SortPairs(nullptr, b1, (const int *)nullptr, (int *)nullptr, (const int *)nullptr,
                                  (int *)nullptr, (int)M, 0, 32, ctx->stream);
  cub::DeviceScan::ExclusiveSum(nullptr, b2, (const int *)nullptr, (int *)nullptr, (int)(E + 1), ctx->stream);
  ctx->cub_bytes = std::max(b1, b2) + 256;
  CUDA_TRY(ctx->cub_tmp.alloc(ctx->cub_bytes));
  return DBL_OK;
}

static int bits_for(int64_t n) {
  int b = 1;
  while (((int64_t)1 << b) < n) ++b;
  return b;
}

// Sort keys of rows a shard does not own must sort behind every real key.  One sentinel value would put 7/8 of the
// items of an 8-rank shard into the same radix bin, and a radix sort serialises on a bin that takes everything; so
// they are spread over the unused top of the key range: `spread` values above n_keys, in a key of `bits` bits.
static void sentinel_spread(int64_t n_keys, int world, int *bits, long long *spread) {
  int b = bits_for(n_keys + 1);
  long long sp = ((long long)1 << b) - n_keys;
  if (world > 1 && sp < 256) { ++b; sp = ((long long)1 << b) - n_keys; }
  *bits = b;
  *spread = world > 1 ? sp : 1;
}

// CSR entity -> linked records in ascending record id (LinksIndex, GU:84-119)
static int build_links_csr(dbl_ctx *ctx, bool commit_newlinks = false) {
  const int64_t R = ctx->R, E = ctx->E;
  size_t tb = ctx->cub_bytes;
  int bits;
  long long spread;
  sentinel_spread(E, ctx->world, &bits, &spread);
  if (commit_newlinks)  // inside a sweep: the draws of the link kernel become the links (unless the sweep was abandoned)
    k_commit_link_keys<<<grid_for(R, 256), 256, 0, ctx->stream>>>(R, ctx->ctl(), ctx->newlink.p, ctx->link.p,
                                                                 ctx->rec_owned.p, (int)E, (int)spread, ctx->link_key.p);
  else
    k_rec_link_keys<<<grid_for(R, 256), 256, 0, ctx->stream>>>(R, ctx->link.p, ctx->rec_owned.p, (int)E, (int)spread,
                                                              ctx->link_key.p);
  CUDA_TRY(cub::DeviceRadixSort::SortPairs(ctx->cub_tmp.p, tb, (const int *)ctx->link_key.p, ctx->link_sorted.p,
                                           (const int *)ctx->iota.p, ctx->rec_by_ent.p, (int)R, 0, bits, ctx->stream));
  k_segment_ptr<<<grid_for(R + 1, 256), 256, 0, ctx->stream>>>(R, (int)E, ctx->link_sorted.p, ctx->ent_rec_ptr.p);
  ctx->launches += 3;
  return DBL_OK;
}

// group entities and records by block (replaces the shuffle, GU:144); the tiled copies of the entity table are built
// on demand by ensure_tiles().  end_of_sweep: this is the last step of a sweep -- the scan kernel also adopts the
// partial summary as the global one (single rank) and counts the sweep.
static int relayout(dbl_ctx *ctx, bool end_of_sweep = false) {
  const int64_t R = ctx->R, E = ctx->E;
  const int P = ctx->P;
  const int pb = bits_for(P + 1);
  size_t tb = ctx->cub_bytes;
  k_block_keys<<<grid_for(std::max(E, R), 256), 256, 0, ctx->stream>>>(E, R, ctx->blk.p, ctx->link.p, ctx->ent_owned.p,
                                                                        ctx->rec_owned.p, ctx->rec_class.p, P,
                                                                        ctx->ent_key.p, ctx->rec_key.p);
  CUDA_TRY(cub::DeviceRadixSort::SortPairs(ctx->cub_tmp.p, tb, (const int *)ctx->ent_key.p, ctx->blk_sorted.p,
                                           (const int *)ctx->iota.p, ctx->ent_sorted.p, (int)E, 0, pb, ctx->stream));
  tb = ctx->cub_bytes;
  CUDA_TRY(cub::DeviceRadixSort::SortPairs(ctx->cub_tmp.p, tb, (const int *)ctx->rec_key.p, ctx->rec_key_sorted.p,
                                           (const int *)ctx->iota.p, ctx->rec_sorted.p, (int)R, 0,
                                           pb + REC_CLASS_BITS, ctx->stream));
  k_block_ptrs<<<grid_for(std::max(E, R) + 1, 256), 256, 0, ctx->stream>>>(E, R, P, ctx->blk_sorted.p, ctx->ent_ptr.p,
                                                                            ctx->rec_key_sorted.p, ctx->rec_ptr.p);
  k_block_scan<<<1, 128, 0, ctx->stream>>>(P, ctx->ent_ptr.p, ctx->rec_ptr.p, ctx->tile_ptr.p, ctx->cta_ptr.p,
                                           LINK_WARPS, ctx->cta_ptr2.p, MATCH_WARPS, ctx->cta_ptr3.p, ctx->pcg2_recs, ctx->ctl(),
                                           (end_of_sweep && ctx->world <= 1) ? ctx->nw : 0, ctx->part(), ctx->glob(),
                                           end_of_sweep ? 1 : 0);
  ctx->launches += 9;
  ctx->inv_valid = false;
  ctx->tiles_valid[0] = ctx->tiles_valid[1] = false;
  ctx->h_owned_ent = ctx->h_owned_rec = -1;  // changed on the device; snapshot() brings them back
  CUDA_TRY(cudaGetLastError());
  return DBL_OK;
}

// tiled copy of the block-sorted entity table in the format the coming link kernel reads (1: attribute-major, 2: quad)
static int ensure_tiles(dbl_ctx *ctx, int fmt) {
  if (ctx->tiles_valid[fmt - 1]) return DBL_OK;
  const int64_t n_slots = (int64_t)((size_t)(ctx->E / TE) + (size_t)ctx->P + 1) * TE;
  k_build_tiles<<<grid_for(n_slots, 256), 256, 0, ctx->stream>>>(n_slots, fmt, ctx->A, ctx->y.p, ctx->entN.p,
                                                                 ctx->ent_sorted.p, ctx->ent_ptr.p, ctx->tile_ptr.p,
                                                                 ctx->tiles.p, ctx->perm_dev.p, ctx->P, ctx->pack_consts,
                                                                 ctx->qtiles.p, ctx->n_str, ctx->qtile_pk);
  ctx->launches += 1;
  ctx->tiles_valid[fmt - 1] = true;
  CUDA_TRY(cudaGetLastError());
  return DBL_OK;
}

// entity N / block ids / partial summary of the owned rows; in_sweep: prefix mode + distortion draws (GU:324-359)
static int refresh_summary(dbl_ctx *ctx, bool in_sweep) {
  const int A = ctx->A, F = ctx->F;
  if (!in_sweep) CUDA_TRY(cudaMemsetAsync(ctx->part(), 0, sizeof(long long) * ctx->nw, ctx->stream));  // else: k_theta
  EntPostParams ep;
  ep.rows = in_sweep ? rows_prefix(ctx, true) : rows_masked(ctx, true);
  ep.A = A; ep.y = ctx->y.p; ep.attrs = ctx->attrs.p; ep.tree = ctx->tree; ep.entN = ctx->entN.p; ep.blk = ctx->blk.p;
  ep.ent_rec_ptr = ctx->ent_rec_ptr.p; ep.part = ctx->part(); ep.iso_slot = ctx->iso_slot(); ep.ll_slot = ctx->ll_slot();
  ep.blk_slot = ctx->world > 1 ? ctx->blk_ent_slot() : -1;
  k_entity_post<<<grid_rows(ctx->E, 256), 256, 0, ctx->stream>>>(ep);
  DistParams dp;
  dp.A = A; dp.F = F; dp.draw = in_sweep ? 1 : 0; dp.seed = ctx->seed;
  dp.rows = in_sweep ? rows_prefix(ctx, false) : rows_masked(ctx, false);
  dp.attrs = ctx->attrs.p; dp.x = ctx->x.p; dp.file = ctx->file.p; dp.link = ctx->link.p;
  dp.y = ctx->y.p; dp.blk = ctx->blk.p; dp.zmask = ctx->zmask.p; dp.theta = ctx->theta(); dp.part = ctx->part();
  dp.ll_slot = ctx->ll_slot();
  dp.blk_slot = ctx->world > 1 ? ctx->blk_rec_slot() : -1;
  k_dist<<<grid_rows(ctx->R, 256), 256, 0, ctx->stream>>>(dp);
  ctx->launches += 3;
  CUDA_TRY(cudaGetLastError());
  return DBL_OK;
}

// the partial summary of a context that owns everything IS the global one
static int adopt_local_summary(dbl_ctx *ctx) {
  k_reduce_local<<<1, 256, 0, ctx->stream>>>(ctx->nw, ctx->ctl(), ctx->part(), ctx->glob());
  ctx->launches += 1;
  CUDA_TRY(cudaGetLastError());
  return DBL_OK;
}

static void recycle_events(dbl_ctx *ctx) {
  for (auto &pe : ctx->pending_events) {
    float ms[4] = {0.f, 0.f, 0.f, 0.f};
    bool ok = true;
    for (int i = 0; i < 4; ++i) ok = ok && cudaEventElapsedTime(&ms[i], pe.e[i], pe.e[i + 1]) == cudaSuccess;
    if (ok) {
      ctx->link_ms += ms[0];
      ctx->link_launches += 1;
      for (int i = 0; i < 4; ++i) ctx->phase_ms[i] += ms[i];
      ctx->phase_sweeps += 1;
    }
    ctx->event_pool.push_back(pe);
  }
  ctx->pending_events.clear();
}

// One device -> host copy of the control block, one synchronisation: iteration, status, owned counts, global
// summary, theta.  This is the only point where the host waits for the device.
static int snapshot(dbl_ctx *ctx) {
  CUDA_TRY(cudaMemcpyAsync(ctx->h_cb, ctx->cb.p, ctx->cb_words * sizeof(long long), cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_TRY(cudaStreamSynchronize(ctx->stream));
  recycle_events(ctx);
  const long long *c = ctx->h_ctl();
  ctx->iteration = c[CTL_ITER];
  ctx->h_pairs = c[CTL_PAIRS];
  ctx->h_owned_ent = c[CTL_OWNED_ENT];
  ctx->h_owned_rec = c[CTL_OWNED_REC];
  const long long st = c[CTL_STATUS];
  if (st) {
    const bool sharded = !ctx->all_owned;
    if (!sharded && st == ST_ZERO_MASS) {
      // the abandoned sweep changed nothing but theta: put the previous values back, the state is the one before it
      std::copy(ctx->h_theta_dev() + (size_t)ctx->A * ctx->F, ctx->h_theta_dev() + 2 * (size_t)ctx->A * ctx->F, ctx->h_theta.begin());
      CUDA_TRY(cudaMemcpyAsync(ctx->theta(), ctx->theta_prev(), sizeof(double) * ctx->A * ctx->F, cudaMemcpyDeviceToDevice,
                               ctx->stream));
    } else {
      ctx->has_state = false;  // shards are no longer at the same iteration: the caller has to upload a state again
    }
    CUDA_TRY(cudaMemsetAsync(ctx->ctl() + CTL_STATUS, 0, sizeof(long long), ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    if (st & ST_PEER_TIMEOUT) { ctx->set_error("a peer rank did not reach the exchange barrier (time-out)"); return DBL_ERR_CUDA; }
    ctx->set_error((st & ST_PEER_ERROR) && !(st & ST_ZERO_MASS) ? "the sweep failed on a peer rank"
                                                                : "zero probability mass in a link draw");
    return (st & ST_ZERO_MASS) ? DBL_ERR_ZERO_MASS : DBL_ERR_CUDA;
  }
  std::copy(ctx->h_theta_dev(), ctx->h_theta_dev() + (size_t)ctx->A * ctx->F, ctx->h_theta.begin());
  return DBL_OK;
}

static int finish_new_state(dbl_ctx *ctx, bool check_state, bool new_records) {
  // range checks on the device, then file sizes (RecordsCache.fileSizes)
  CUDA_TRY(cudaMemsetAsync(ctx->vflag.p, 0, sizeof(int), ctx->stream));
  k_validate<<<grid_for(std::max(ctx->R, ctx->E), 256), 256, 0, ctx->stream>>>(
      ctx->R, ctx->E, ctx->A, ctx->F, ctx->attrs.p, ctx->x.p, ctx->file.p, check_state ? ctx->link.p : nullptr,
      check_state ? ctx->y.p : nullptr, ctx->vflag.p);
  int bad = 0;
  CUDA_TRY(cudaMemcpyAsync(&bad, ctx->vflag.p, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  std::vector<int> hc(ctx->F);
  if (new_records) {
    CUDA_TRY(cudaMemsetAsync(ctx->file_cnt.p, 0, sizeof(int) * ctx->F, ctx->stream));
    k_hist<<<grid_for(ctx->R, 256), 256, 0, ctx->stream>>>(ctx->R, ctx->file.p, ctx->file_cnt.p);
    CUDA_TRY(cudaMemcpyAsync(hc.data(), ctx->file_cnt.p, sizeof(int) * ctx->F, cudaMemcpyDeviceToHost, ctx->stream));
  }
  CUDA_TRY(cudaStreamSynchronize(ctx->stream));  // nothing below may run on out-of-range ids
  if (bad) {
    ctx->has_state = false;
    ctx->set_error(bad & 1 ? "record value id out of range" : bad & 2 ? "file id out of range"
                   : bad & 4 ? "link out of range" : "entity value id out of range");
    return DBL_ERR_INVALID;
  }
  if (new_records) {
    ctx->file_sizes.assign(hc.begin(), hc.end());
    ctx->h_file_sizes_d.assign(hc.begin(), hc.end());
    CUDA_TRY(cudaMemcpyAsync(ctx->prior.p + 2 * ctx->A, ctx->h_file_sizes_d.data(), sizeof(double) * ctx->F,
                             cudaMemcpyHostToDevice, ctx->stream));
  }
  ctx->launches += 2;
  // iteration / status of the new state
  ctx->h_head[0] = ctx->iteration; ctx->h_head[1] = 0;
  CUDA_TRY(cudaMemcpyAsync(ctx->ctl(), ctx->h_head, sizeof(ctx->h_head), cudaMemcpyHostToDevice, ctx->stream));
  int rc = build_links_csr(ctx);
  if (rc) return rc;
  rc = refresh_summary(ctx, false);
  if (rc) return rc;
  rc = adopt_local_summary(ctx);
  if (rc) return rc;
  // a sharded context is carved up by dbl_set_block_owners next, which lays the shard out; until then nothing reads
  // the layout (dbl_set_partitioner builds its own)
  if (ctx->world <= 1) {
    rc = relayout(ctx);
    if (rc) return rc;
  }
  rc = snapshot(ctx);
  if (rc) return rc;
  ctx->has_state = true;
  return DBL_OK;
}

extern "C" int dbl_set_partitioner(dbl_ctx *ctx, const dbl_kdtree *tree) {
  if (!ctx) return DBL_ERR_INVALID;
  CUDA_TRY(cudaSetDevice(ctx->device));
  CUDA_TRY(cudaStreamSynchronize(ctx->stream));
  if (ctx->has_state && !ctx->all_owned) { ctx->set_error("dbl_set_partitioner after dbl_set_block_owners"); return DBL_ERR_STATE; }
  ctx->drop_graphs();
  int rc = upload_tree(ctx, tree);
  if (rc) return rc;
  if (!ctx->has_state) return alloc_control(ctx);
  rc = alloc_blocks(ctx);
  if (rc) return rc;
  rc = refresh_summary(ctx, false);  // recomputes block ids (and the unchanged summary)
  if (rc) return rc;
  rc = adopt_local_summary(ctx);
  if (rc) return rc;
  rc = relayout(ctx);
  if (rc) return rc;
  return snapshot(ctx);
}
extern "C" int32_t dbl_num_partitions(const dbl_ctx *ctx) { return ctx ? ctx->P : 0; }

static int upload_theta(dbl_ctx *ctx) {
  const size_t n = (size_t)ctx->A * ctx->F;
  CUDA_TRY(cudaMemcpyAsync(ctx->theta(), ctx->h_theta.data(), sizeof(double) * n, cudaMemcpyHostToDevice, ctx->stream));
  CUDA_TRY(cudaMemcpyAsync(ctx->theta_prev(), ctx->h_theta.data(), sizeof(double) * n, cudaMemcpyHostToDevice, ctx->stream));
  return DBL_OK;  // h_theta is next written by snapshot(), i.e. after the stream has drained
}

extern "C" int dbl_state_init(dbl_ctx *ctx, int64_t R, const int32_t *x, const int32_t *file, int64_t pop) {
  if (!ctx || !x || !file) return DBL_ERR_INVALID;
  CUDA_TRY(cudaSetDevice(ctx->device));
  const int64_t E = pop > 0 ? pop : R;
  int rc = alloc_state(ctx, R, E);
  if (rc) return rc;
  const int A = ctx->A;
  CUDA_TRY(cudaMemcpyAsync(ctx->x.p, x, sizeof(int) * R * A, cudaMemcpyHostToDevice, ctx->stream));
  k_rec_class<<<grid_for(R, 256), 256, 0, ctx->stream>>>(R, A, ctx->attrs.p, ctx->x.p, ctx->rec_class.p);
  CUDA_TRY(cudaMemcpyAsync(ctx->file.p, file, sizeof(int) * R, cudaMemcpyHostToDevice, ctx->stream));
  k_init_entities<<<grid_for(E * A, 256), 256, 0, ctx->stream>>>(E, R, A, ctx->seed, ctx->attrs.p, ctx->x.p, ctx->y.p);
  k_init_records<<<grid_for(R, 256), 256, 0, ctx->stream>>>(E, R, A, ctx->x.p, ctx->y.p, ctx->link.p, ctx->zmask.p);
  ctx->launches += 3;
  for (int a = 0; a < A; ++a)
    for (int f = 0; f < ctx->F; ++f)
      ctx->h_theta[a * ctx->F + f] = ctx->alpha[a] / (ctx->alpha[a] + ctx->beta[a]);  // DistortionProbs.scala:38-40
  rc = upload_theta(ctx);
  if (rc) return rc;
  ctx->iteration = 0;
  return finish_new_state(ctx, false, true);
}

extern "C" int dbl_state_upload(dbl_ctx *ctx, int64_t R, int64_t E, const int32_t *x, const int32_t *file,
                                const uint8_t *z, const int32_t *link, const int32_t *y, const double *theta,
                                int64_t iteration) {
  if (!ctx || !z || !link || !y || !theta || ((x == nullptr) != (file == nullptr))) return DBL_ERR_INVALID;
  const bool new_records = (x != nullptr);
  if (!new_records && (!ctx->x.p || ctx->R != R || ctx->E != E)) {
    ctx->set_error("dbl_state_upload without records: the context holds no records / state of that shape");
    return DBL_ERR_STATE;
  }
  CUDA_TRY(cudaSetDevice(ctx->device));
  int rc = alloc_state(ctx, R, E);
  if (rc) return rc;
  const int A = ctx->A;
  DevBuf<uint8_t> &zb = ctx->zbytes;
  if (new_records) {
    CUDA_TRY(cudaMemcpyAsync(ctx->x.p, x, sizeof(int) * R * A, cudaMemcpyDefault, ctx->stream));
    k_rec_class<<<grid_for(R, 256), 256, 0, ctx->stream>>>(R, A, ctx->attrs.p, ctx->x.p, ctx->rec_class.p);
    CUDA_TRY(cudaMemcpyAsync(ctx->file.p, file, sizeof(int) * R, cudaMemcpyDefault, ctx->stream));
  }
  CUDA_TRY(cudaMemcpyAsync(zb.p, z, (size_t)R * A, cudaMemcpyDefault, ctx->stream));
  CUDA_TRY(cudaMemcpyAsync(ctx->link.p, link, sizeof(int) * R, cudaMemcpyDefault, ctx->stream));
  CUDA_TRY(cudaMemcpyAsync(ctx->y.p, y, sizeof(int) * E * A, cudaMemcpyDefault, ctx->stream));
  k_pack_z<<<grid_for(R, 256), 256, 0, ctx->stream>>>(R, A, zb.p, ctx->zmask.p);
  ctx->launches += 2;
  std::copy(theta, theta + (size_t)A * ctx->F, ctx->h_theta.begin());
  rc = upload_theta(ctx);
  if (rc) return rc;
  ctx->iteration = iteration;
  return finish_new_state(ctx, true, new_records);
}

extern "C" int dbl_state_download(dbl_ctx *ctx, uint8_t *z, int32_t *link, int32_t *y, double *theta,
                                  int32_t *block_of_entity) {
  if (!ctx) return DBL_ERR_INVALID;
  if (!ctx->has_state) { ctx->set_error("no state"); return DBL_ERR_STATE; }
  CUDA_TRY(cudaSetDevice(ctx->device));
  const int A = ctx->A;
  DevBuf<uint8_t> &zb = ctx->zbytes;
  if (z) {
    k_unpack_z<<<grid_for(ctx->R, 256), 256, 0, ctx->stream>>>(ctx->R, A, ctx->zmask.p, zb.p);
    ctx->launches += 1;
    CUDA_TRY(cudaMemcpyAsync(z, zb.p, (size_t)ctx->R * A, cudaMemcpyDeviceToHost, ctx->stream));
  }
  if (link) CUDA_TRY(cudaMemcpyAsync(link, ctx->link.p, sizeof(int) * ctx->R, cudaMemcpyDeviceToHost, ctx->stream));
  if (y) CUDA_TRY(cudaMemcpyAsync(y, ctx->y.p, sizeof(int) * ctx->E * A, cudaMemcpyDeviceToHost, ctx->stream));
  if (block_of_entity)
    CUDA_TRY(cudaMemcpyAsync(block_of_entity, ctx->blk.p, sizeof(int) * ctx->E, cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_TRY(cudaStreamSynchronize(ctx->stream));
  if (theta) std::copy(ctx->h_theta.begin(), ctx->h_theta.end(), theta);
  return DBL_OK;
}

extern "C" int dbl_links_download(dbl_ctx *ctx, int32_t *link_out, int32_t *block_out) {
  return dbl_state_download(ctx, nullptr, link_out, nullptr, nullptr, block_out);
}

// ---------------------------------------------------------------------------------------------------
// link kernel dispatch
// ---------------------------------------------------------------------------------------------------
#define DBL_DECL(N) int dbl_launch_pcg2_a##N(int ns, int grid, cudaStream_t stream, const LinkParams &lp, size_t *cfg);
DBL_DECL(1) DBL_DECL(2) DBL_DECL(3) DBL_DECL(4) DBL_DECL(5) DBL_DECL(6) DBL_DECL(7) DBL_DECL(8)
DBL_DECL(9) DBL_DECL(10) DBL_DECL(11) DBL_DECL(12) DBL_DECL(13) DBL_DECL(14) DBL_DECL(15) DBL_DECL(16)
#undef DBL_DECL

// number of entities in owned blocks, on the host.  Unsharded contexts own everything; otherwise the count lives on
// the device (the exchange changes it every sweep) and costs one small read-back.
static int owned_entities_on_host(dbl_ctx *ctx, int64_t *out) {
  if (ctx->all_owned && !ctx->in_block_sweep) { *out = ctx->E; return DBL_OK; }
  if (ctx->h_owned_ent < 0) {
    long long v = 0;
    CUDA_TRY(cudaMemcpyAsync(&v, ctx->ctl() + CTL_OWNED_ENT, sizeof(v), cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    ctx->h_owned_ent = v;
  }
  *out = ctx->h_owned_ent;
  return DBL_OK;
}

// (block, attribute, value) -> candidate positions, for k_link_pruned
static int ensure_inverted_index(dbl_ctx *ctx) {
  if (ctx->inv_valid) return DBL_OK;
  const int64_t cap = ctx->E * ctx->A;
  if (cap > 0x7fffffff) { ctx->set_error("inverted index too large"); return DBL_ERR_INVALID; }
  InvDense &dn = ctx->inv_dense;
  dn.A = ctx->A; dn.sumV = 0;
  for (int k = 0; k < ctx->A; ++k) { dn.voff[k] = dn.sumV; dn.sumV += ctx->h_attrs[ctx->perm[k]].V; }
  const long long n_ids = (long long)ctx->P * dn.sumV;
  long long dense_max = 1ll << 25;  // entries; DBL_INV_DENSE_MAX overrides (tests force the binary-search path with 0)
  if (const char *ev = getenv("DBL_INV_DENSE_MAX")) dense_max = atoll(ev);
  ctx->inv_use_dense = n_ids <= dense_max;
  int vmax = 1;
  for (int a = 0; a < ctx->A; ++a) vmax = std::max(vmax, ctx->h_attrs[a].V);
  ctx->inv_vbits = bits_for(vmax + 1);
  dn.vbits = ctx->inv_vbits;

  if (ctx->inv_use_dense) {
    // dense (block, attribute, value) -> posting pointers: the table is small enough (P * sum of vocabulary sizes
    // entries).  32-bit keys (the dense id), every slot of the sorted table sorted (non-owned rows carry the
    // sentinel id): no size depends on the shard, nothing is read back.
    if (ctx->inv_key32.n != (size_t)cap) {
      CUDA_TRY(ctx->inv_key32_in.alloc(cap));
      CUDA_TRY(ctx->inv_key32.alloc(cap));
      if (ctx->inv_pos.n != (size_t)cap) { CUDA_TRY(ctx->inv_pos_in.alloc(cap)); CUDA_TRY(ctx->inv_pos.alloc(cap)); }
      size_t tb = 0;
      cub::DeviceRadixSort::SortPairs(nullptr, tb, (const unsigned *)nullptr, (unsigned *)nullptr, (const int *)nullptr,
                                      (int *)nullptr, (int)cap, 0, 32, ctx->stream);
      if (ctx->inv_tmp_bytes < tb + 256) { ctx->inv_tmp_bytes = tb + 256; CUDA_TRY(ctx->inv_tmp.alloc(ctx->inv_tmp_bytes)); }
    }
    if (ctx->inv_vptr.n != (size_t)n_ids + 1) CUDA_TRY(ctx->inv_vptr.alloc((size_t)n_ids + 1));
    int ibits;
    long long ispread;
    sentinel_spread(n_ids, ctx->world, &ibits, &ispread);
    k_inv_keys32<<<grid_for(cap, 256), 256, 0, ctx->stream>>>(ctx->E, ctx->A, ctx->P, dn, n_ids, ispread, ctx->y.p,
                                                             ctx->blk_sorted.p, ctx->ent_sorted.p, ctx->ent_ptr.p,
                                                             ctx->perm_dev.p, ctx->inv_key32_in.p, ctx->inv_pos_in.p);
    size_t tb = ctx->inv_tmp_bytes;
    // stable radix sort on the significant bits only: positions stay ascending inside a key
    CUDA_TRY(cub::DeviceRadixSort::SortPairs(ctx->inv_tmp.p, tb, (const unsigned *)ctx->inv_key32_in.p, ctx->inv_key32.p,
                                             (const int *)ctx->inv_pos_in.p, ctx->inv_pos.p, (int)cap, 0,
                                             ibits, ctx->stream));
    k_inv_value_ptr32<<<grid_for(cap + 1, 256), 256, 0, ctx->stream>>>(cap, n_ids, (long long)dn.sumV, ctx->inv_key32.p,
                                                                       ctx->inv_vptr.p);
    ctx->launches += 5;
    ctx->inv_valid = true;
    CUDA_TRY(cudaGetLastError());
    return DBL_OK;
  }

  // too many (block, attribute, value) ids for a dense table: 64-bit keys ((block, attribute) group | value) over the
  // entities of owned blocks (they come first in ent_sorted), (block, attribute) segment pointers, and a binary
  // search per record.  The owned count sizes the sort, so a sharded context reads it back once per sweep.
  int64_t owned = 0;
  { int rc = owned_entities_on_host(ctx, &owned); if (rc) return rc; }
  const int64_t n = owned * ctx->A;
  if (ctx->inv_key.n != (size_t)cap) {
    CUDA_TRY(ctx->inv_key_in.alloc(cap));
    CUDA_TRY(ctx->inv_key.alloc(cap));
    if (ctx->inv_pos.n != (size_t)cap) { CUDA_TRY(ctx->inv_pos_in.alloc(cap)); CUDA_TRY(ctx->inv_pos.alloc(cap)); }
    size_t tb = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, tb, (const unsigned long long *)nullptr, (unsigned long long *)nullptr,
                                    (const int *)nullptr, (int *)nullptr, (int)cap, 0, 64, ctx->stream);
    if (ctx->inv_tmp_bytes < tb + 256) { ctx->inv_tmp_bytes = tb + 256; CUDA_TRY(ctx->inv_tmp.alloc(ctx->inv_tmp_bytes)); }
  }
  const int nbits = ctx->inv_vbits + bits_for((int64_t)(ctx->P + 1) * ctx->A);
  if (n > 0) {
    k_inv_keys<<<grid_for(n, 256), 256, 0, ctx->stream>>>(owned, ctx->A, ctx->P, ctx->inv_vbits,
                                                          ctx->y.p, ctx->blk_sorted.p, ctx->ent_sorted.p,
                                                          ctx->ent_ptr.p, ctx->perm_dev.p, ctx->inv_key_in.p,
                                                          ctx->inv_pos_in.p);
    size_t tb = ctx->inv_tmp_bytes;
    CUDA_TRY(cub::DeviceRadixSort::SortPairs(ctx->inv_tmp.p, tb, (const unsigned long long *)ctx->inv_key_in.p,
                                             ctx->inv_key.p, (const int *)ctx->inv_pos_in.p, ctx->inv_pos.p, (int)n,
                                             0, std::min(64, nbits), ctx->stream));
  }
  const int n_groups = (ctx->P + 1) * ctx->A;
  if (ctx->inv_seg.n != (size_t)n_groups + 1) CUDA_TRY(ctx->inv_seg.alloc((size_t)n_groups + 1));
  k_inv_segments<<<grid_for(n + 1, 256), 256, 0, ctx->stream>>>(n, n_groups, ctx->inv_vbits, ctx->inv_key.p,
                                                                ctx->inv_seg.p);
  ctx->launches += 5;
  ctx->inv_valid = true;
  CUDA_TRY(cudaGetLastError());
  return DBL_OK;
}

static bool pcg2_kernel_fits(const dbl_ctx *ctx) {
  return ctx->hslots > 0 && ctx->A <= LINK_MAX_UNROLL_A &&
         pcg2_smem_bytes(ctx->A, ctx->n_str, ctx->hslots, ctx->qtile_pk != 0) <= 100 * 1024;
}
static int dispatch_pcg2(dbl_ctx *ctx, int grid, const LinkParams &lp) {
  int rc = -1;
  switch (ctx->A) {
#define DBL_CASE(N) case N: rc = dbl_launch_pcg2_a##N(ctx->n_str, grid, ctx->stream, lp, &ctx->pcg2_smem_cfg); break;
    DBL_CASE(1) DBL_CASE(2) DBL_CASE(3) DBL_CASE(4) DBL_CASE(5) DBL_CASE(6) DBL_CASE(7) DBL_CASE(8)
    DBL_CASE(9) DBL_CASE(10) DBL_CASE(11) DBL_CASE(12) DBL_CASE(13) DBL_CASE(14) DBL_CASE(15) DBL_CASE(16)
#undef DBL_CASE
  }
  if (rc != 0) { ctx->set_error(std::string("k_link_pcg2 launch: ") + cudaGetErrorString((cudaError_t)rc)); return DBL_ERR_CUDA; }
  return DBL_OK;
}

static int launch_link(dbl_ctx *ctx, int sampler) {
  const int A = ctx->A;
  LinkParams lp;
  memset(&lp, 0, sizeof(lp));
  lp.A = A; lp.F = ctx->F; lp.P = ctx->P; lp.sampler = sampler; lp.seed = ctx->seed; lp.ctl = ctx->ctl();
  lp.attrs = ctx->attrs.p; lp.x = ctx->x.p; lp.file = ctx->file.p; lp.link = ctx->link.p; lp.zmask = ctx->zmask.p;
  lp.theta = ctx->theta(); lp.ent_ptr = ctx->ent_ptr.p; lp.tile_ptr = ctx->tile_ptr.p; lp.rec_ptr = ctx->rec_ptr.p;
  lp.cta_ptr = ctx->cta_ptr.p; lp.ent_sorted = ctx->ent_sorted.p; lp.rec_sorted = ctx->rec_sorted.p;
  lp.tiles = ctx->tiles.p; lp.newlink = ctx->newlink.p;
  lp.qtiles = ctx->qtiles.p; lp.qtile_pk = ctx->qtile_pk;
  lp.work = reinterpret_cast<unsigned long long *>(ctx->ctl() + CTL_WORK);
  lp.lane_sums = ctx->lane_sums.p;
  lp.status = reinterpret_cast<unsigned long long *>(ctx->ctl() + CTL_STATUS);
  lp.pairs = reinterpret_cast<unsigned long long *>(ctx->ctl() + CTL_PAIRS);
  for (int k = 0; k < A; ++k) lp.perm[k] = ctx->perm[k];
  lp.blk_of_link = ctx->blk.p;
  lp.pack_consts = ctx->pack_consts;
  const size_t ring = (size_t)LINK_STAGES * tile_words(A) * 4 + 128;
  const int mode = ctx->link_mode;  // 0 auto, 1 force generic
  lp.hslots = ctx->hslots; lp.hshift = ctx->hshift;
  if (mode != 1 && sampler == DBL_PCG_II && pcg2_kernel_fits(ctx)) {
    // persistent CTAs: a few per SM, each takes groups of LINK_WARPS records from the work counter until none is left
    // (k_theta zeroed the counter; the block-level API launches the kernel once per block after one k_theta)
    if (ctx->in_block_sweep) CUDA_TRY(cudaMemsetAsync(lp.work, 0, sizeof(unsigned long long), ctx->stream));
    int rc = ensure_tiles(ctx, 2);
    if (rc) return rc;
    lp.cta_ptr = ctx->cta_ptr3.p;  // work items of PCG2_RECS records
    return dispatch_pcg2(ctx, std::min(ctx->max_ctas, ctx->pcg2_grid), lp);
  }
  {
    int rc = ensure_tiles(ctx, 1);  // every other link kernel reads the attribute-major tiles
    if (rc) return rc;
  }
  if (mode == 0 && sampler != DBL_PCG_II) {  // pruned scoring through the inverted index
    int rc = ensure_inverted_index(ctx);
    if (rc) return rc;
    int64_t owned = 0;
    if (!ctx->inv_use_dense) {
      rc = owned_entities_on_host(ctx, &owned);
      if (rc) return rc;
    }
    PrunedParams pp;
    pp.lp = lp;
    pp.inv_key = ctx->inv_key.p;
    pp.inv_pos = ctx->inv_pos.p;
    pp.inv_n = (long long)owned * ctx->A;
    pp.R = ctx->R;
    pp.vbits = ctx->inv_vbits;
    pp.inv_seg = ctx->inv_seg.p;
    pp.rec_key_sorted = ctx->rec_key_sorted.p;
    pp.rec_key_shift = REC_CLASS_BITS;
    pp.inv_vptr = ctx->inv_use_dense ? ctx->inv_vptr.p : nullptr;
    pp.sumV = ctx->inv_dense.sumV;
    for (int k = 0; k < A; ++k) pp.voff[k] = ctx->inv_dense.voff[k];
    if (ctx->heavy_list.n != (size_t)ctx->R) CUDA_TRY(ctx->heavy_list.alloc((size_t)ctx->R));
    pp.heavy_list = ctx->heavy_list.p;
    if (ctx->in_block_sweep)  // the block-level API launches once per block after one k_theta
      CUDA_TRY(cudaMemsetAsync(ctx->ctl() + CTL_HEAVY, 0, sizeof(long long), ctx->stream));
    k_link_pruned<<<(int)std::min<int64_t>(grid_for(ctx->R, LINK_WARPS), (int64_t)ctx->sm_count * 16), LINK_WARPS * 32, 0,
                    ctx->stream>>>(pp);
    // records whose whole block has to be scored (no must-match attribute), a CTA each; usually none: the kernel
    // reads the count and returns
    k_link_heavy<<<ctx->sm_count * 2, HEAVY_WARPS * 32, 0, ctx->stream>>>(pp);
    ctx->launches += 1;
    return DBL_OK;
  }
  if (mode != 1 && sampler != DBL_PCG_II && ring <= 160 * 1024) {
    if (ctx->match_smem_cfg < ring) {
      CUDA_TRY(cudaFuncSetAttribute(k_link_match, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ring));
      ctx->match_smem_cfg = ring;
    }
    lp.cta_ptr = ctx->cta_ptr2.p;  // MATCH_WARPS records per CTA
    const int grid = (int)((ctx->R + MATCH_WARPS - 1) / MATCH_WARPS) + ctx->P;
    k_link_match<<<grid, (MATCH_WARPS + 1) * 32, ring, ctx->stream>>>(lp);
    return DBL_OK;
  }
  k_link_generic<<<ctx->max_ctas, LINK_WARPS * 32, 0, ctx->stream>>>(lp);
  return DBL_OK;
}

// ---------------------------------------------------------------------------------------------------
// one application of State.nextState (State.scala:78-99), enqueued on the context's stream without any host
// synchronisation (PCG-II; the pruned PCG-I kernel of a SHARDED context reads one count back per sweep)
// ---------------------------------------------------------------------------------------------------
// (1) theta | summary of the previous state (State.scala:83, GU:305-320)
static int enqueue_theta(dbl_ctx *ctx) {
  k_theta<<<1, 128, 0, ctx->stream>>>(ctx->A, ctx->F, ctx->seed, ctx->ctl(), ctx->glob(), ctx->prior.p,
                                       ctx->prior.p + ctx->A, ctx->prior.p + 2 * ctx->A, ctx->theta(), ctx->theta_prev(),
                                       ctx->part(), ctx->nw);
  ctx->launches += 1;
  CUDA_TRY(cudaGetLastError());
  return DBL_OK;
}

// (2)-(4) for the owned entities / records (all of them on an unsharded context): updatePartition, GU:156-211
static int update_owned(dbl_ctx *ctx, int sampler) {
  const int A = ctx->A, F = ctx->F;
  // (2) links
  const bool timed = ctx->cur_timed;
  if (timed) CUDA_TRY(cudaEventRecord(ctx->cur_events.e[0], ctx->stream));
  {
    int rc = launch_link(ctx, sampler);
    if (rc) return rc;
  }
  if (timed) CUDA_TRY(cudaEventRecord(ctx->cur_events.e[1], ctx->stream));
  ctx->launches += 1;
  CUDA_TRY(cudaGetLastError());
  // (3) entity values (the links are committed by the first kernel of the CSR build)
  int rc = build_links_csr(ctx, true);
  if (rc) return rc;
  ValParams vp;
  vp.A = A; vp.F = F; vp.sampler = sampler; vp.seed = ctx->seed; vp.rows = rows_prefix(ctx, true);
  vp.attrs = ctx->attrs.p; vp.x = ctx->x.p; vp.file = ctx->file.p; vp.zmask = ctx->zmask.p; vp.theta = ctx->theta();
  vp.ent_rec_ptr = ctx->ent_rec_ptr.p; vp.rec_by_ent = ctx->rec_by_ent.p; vp.y = ctx->y.p;
  // latency-bound sizes (the grid does not fill the GPU a few times over): the variant with batched loads
  if (ctx->E * A <= (int64_t)ctx->sm_count * 2048 * 4) k_values<8><<<grid_rows(ctx->E * A, 128), 128, 0, ctx->stream>>>(vp);
  else k_values<DBL_VALUES_UB_LARGE><<<grid_rows(ctx->E * A, 128), 128, 0, ctx->stream>>>(vp);
  k_values_log<<<std::min(grid_rows(ctx->E * A, 128), ctx->sm_count * 4), 128, 0, ctx->stream>>>(vp);
  ctx->launches += 2;
  // (4) N(e), new block ids, distortions, partial summary
  return refresh_summary(ctx, true);
}

// (5) the shuffle (GU:144) + the global summary (SummaryAccumulators.scala:54-63), peer to peer
static int exchange_p2p(dbl_ctx *ctx) {
  MoveParams mp;
  mp.c = ctx->comm; mp.ctl = ctx->ctl(); mp.A = ctx->A; mp.ent_sorted = ctx->ent_sorted.p; mp.rec_sorted = ctx->rec_sorted.p;
  mp.blk = ctx->blk.p; mp.owner = ctx->owner.p; mp.link = ctx->link.p; mp.y = ctx->y.p; mp.zmask = ctx->zmask.p;
  mp.ent_dest = ctx->ent_dest.p; mp.ent_owned = ctx->ent_owned.p; mp.rec_owned = ctx->rec_owned.p;
  k_move_ent<<<grid_rows(ctx->E, 256), 256, 0, ctx->stream>>>(mp);
  k_move_rec<<<grid_rows(ctx->R, 256), 256, 0, ctx->stream>>>(mp);
  k_publish_barrier<<<1, 256, 0, ctx->stream>>>(ctx->comm, ctx->ctl(), ctx->part(), ctx->nw, ctx->barrier_timeout_cycles);
  UnpackParams up;
  up.c = ctx->comm; up.ctl = ctx->ctl(); up.A = ctx->A; up.attrs = ctx->attrs.p; up.tree = ctx->tree; up.y = ctx->y.p;
  up.blk = ctx->blk.p; up.link = ctx->link.p; up.entN = ctx->entN.p; up.zmask = ctx->zmask.p;
  up.ent_owned = ctx->ent_owned.p; up.rec_owned = ctx->rec_owned.p;
  k_unpack_ent_p2p<<<grid_rows(ctx->E, 256), 256, 0, ctx->stream>>>(up);
  k_unpack_rec_p2p<<<grid_rows(ctx->R, 256), 256, 0, ctx->stream>>>(up);
  k_reduce_peers<<<1, 256, 0, ctx->stream>>>(ctx->comm, ctx->ctl(), ctx->nw, ctx->ll_slot(), ctx->glob());
  ctx->launches += 6;
  if (ctx->rebalance_period > 0 && ctx->P <= 1024) {
    k_lpt<<<1, 32, 0, ctx->stream>>>(ctx->P, ctx->world, ctx->blk_ent_slot(), ctx->blk_rec_slot(), ctx->glob(), ctx->ctl(),
                                     ctx->rebalance_period, ctx->rebalance_threshold, ctx->owner.p, ctx->lpt_scratch.p,
                                     ctx->lpt_dscratch.p);
    ctx->launches += 1;
  }
  CUDA_TRY(cudaGetLastError());
  return DBL_OK;
}

static int enqueue_sweep_phases(dbl_ctx *ctx, int sampler) {
  const bool timed = ctx->cur_timed;
  int rc = enqueue_theta(ctx);
  if (rc) return rc;
  rc = update_owned(ctx, sampler);
  if (rc) return rc;
  if (timed) CUDA_TRY(cudaEventRecord(ctx->cur_events.e[2], ctx->stream));
  if (ctx->world > 1) {
    rc = exchange_p2p(ctx);
    if (rc) return rc;
  }
  if (timed) CUDA_TRY(cudaEventRecord(ctx->cur_events.e[3], ctx->stream));
  rc = relayout(ctx, true);  // + global summary of a single rank, + iteration count
  if (rc) return rc;
  if (timed) CUDA_TRY(cudaEventRecord(ctx->cur_events.e[4], ctx->stream));
  return DBL_OK;
}

static int enqueue_sweep(dbl_ctx *ctx, int sampler) {
  ctx->cur_timed = !ctx->capturing && ctx->pending_events.size() < 256;  // per-phase timing (eager sweeps only)
  if (ctx->cur_timed) {
    if (!ctx->event_pool.empty()) { ctx->cur_events = ctx->event_pool.back(); ctx->event_pool.pop_back(); }
    else for (cudaEvent_t &e : ctx->cur_events.e) CUDA_TRY(cudaEventCreate(&e));
  }
  const int rc = enqueue_sweep_phases(ctx, sampler);
  if (ctx->cur_timed) (rc ? ctx->event_pool : ctx->pending_events).push_back(ctx->cur_events);
  ctx->cur_timed = false;
  return rc;
}

static int check_sweep_args(dbl_ctx *ctx, int sampler, int32_t n_sweeps) {
  if (sampler < 0 || sampler > 3 || n_sweeps < 0) { ctx->set_error("bad sampler / n_sweeps"); return DBL_ERR_INVALID; }
  if (!ctx->has_state) { ctx->set_error("dbl_sweep before dbl_state_init/upload"); return DBL_ERR_STATE; }
  if (ctx->world > 1 && !ctx->comm_ready) {
    ctx->set_error("dbl_sweep on a sharded context needs dbl_comm_export / dbl_comm_import first "
                   "(or drive the host-mediated exchange: dbl_sweep_begin / dbl_exchange_* / dbl_sweep_end)");
    return DBL_ERR_STATE;
  }
  if (ctx->world > 1 && ctx->all_owned) { ctx->set_error("dbl_sweep on a sharded context before dbl_set_block_owners"); return DBL_ERR_STATE; }
  if (ctx->in_sweep) { ctx->set_error("dbl_sweep inside an open sweep"); return DBL_ERR_STATE; }
  return DBL_OK;
}

// Launch-bound sizes (RLdata-sized problems: a sweep is ~50 tiny kernels) replay one captured sweep instead of
// enqueueing it again: nothing in a sweep depends on the host, every varying quantity is read from device memory.
static bool graph_allowed(const dbl_ctx *ctx, int sampler) {
  if (ctx->graph_mode == 1) return false;
  // the pruned link update of a SHARDED context without the dense posting table reads the owned-entity count back
  // every sweep (it sizes a sort)
  if (ctx->world > 1 && sampler != DBL_PCG_II && ctx->link_mode == 0 && !ctx->inv_use_dense) return false;
  if (ctx->graph_mode == 2) return true;
  // PCG-II at large sizes: tens of milliseconds of GPU time per sweep hide the ~35 launches.  The pruned samplers
  // do not: their sweep is ~3 ms of GPU time at 1 M records and shrinks with the rank count while the host's share
  // (launches, CUB set-up) does not -- measured on 8 GPUs with 8 processes on a 16-CPU quota: 280 sweeps/s eagerly
  // (430 on 4 GPUs), host-bound.
  return ctx->R + ctx->E <= 400000 || sampler != DBL_PCG_II;
}

static int run_sweeps(dbl_ctx *ctx, int sampler, int32_t n_sweeps) {
  int s = 0;
  if (n_sweeps >= 2 && graph_allowed(ctx, sampler)) {
    const int key = sampler * 4 + ctx->link_mode;
    if (!ctx->graph_warm[key]) {  // first sweep of this kind eagerly: allocations and opt-ins happen outside a capture
      int rc = enqueue_sweep(ctx, sampler);
      if (rc) return rc;
      ctx->graph_warm[key] = true;
      s = 1;
    }
    auto it = ctx->graphs.find(key);
    if (it == ctx->graphs.end() && n_sweeps - s >= 2) {
      dbl_ctx::SweepGraph g;
      const int64_t before = ctx->launches;
      CUDA_TRY(cudaStreamBeginCapture(ctx->stream, cudaStreamCaptureModeThreadLocal));
      ctx->capturing = true;
      int rc = enqueue_sweep(ctx, sampler);
      ctx->capturing = false;
      cudaError_t e = cudaStreamEndCapture(ctx->stream, &g.graph);
      g.launches = ctx->launches - before;
      ctx->launches = before;
      if (rc) { if (g.graph) cudaGraphDestroy(g.graph); return rc; }
      if (e != cudaSuccess) { ctx->set_error(std::string("graph capture: ") + cudaGetErrorString(e)); return DBL_ERR_CUDA; }
      CUDA_TRY(cudaGraphInstantiate(&g.exec, g.graph, 0));
      it = ctx->graphs.emplace(key, g).first;
    }
    if (it != ctx->graphs.end())
      for (; s < n_sweeps; ++s) {
        CUDA_TRY(cudaGraphLaunch(it->second.exec, ctx->stream));
        ctx->launches += it->second.launches;
      }
  }
  for (; s < n_sweeps; ++s) {
    int rc = enqueue_sweep(ctx, sampler);
    if (rc) return rc;
  }
  return DBL_OK;
}

extern "C" int dbl_sweep_async(dbl_ctx *ctx, int sampler, int32_t n_sweeps) {
  if (!ctx) return DBL_ERR_INVALID;
  int rc = check_sweep_args(ctx, sampler, n_sweeps);
  if (rc) return rc;
  CUDA_TRY(cudaSetDevice(ctx->device));
  if (!ctx->async_open) CUDA_TRY(cudaEventRecord(ctx->ev0, ctx->stream));
  ctx->async_open = true;
  return run_sweeps(ctx, sampler, n_sweeps);
}

extern "C" int dbl_set_graph_mode(dbl_ctx *ctx, int mode) {
  if (!ctx || mode < 0 || mode > 2) return DBL_ERR_INVALID;
  ctx->graph_mode = mode;
  return DBL_OK;
}

extern "C" int dbl_sync(dbl_ctx *ctx) {
  if (!ctx) return DBL_ERR_INVALID;
  if (!ctx->has_state) { ctx->set_error("no state"); return DBL_ERR_STATE; }
  CUDA_TRY(cudaSetDevice(ctx->device));
  const bool timed = ctx->async_open;
  if (timed) CUDA_TRY(cudaEventRecord(ctx->ev1, ctx->stream));
  ctx->async_open = false;
  int rc = snapshot(ctx);
  if (timed) {
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1) == cudaSuccess) ctx->last_sweep_ms = ms;
  }
  return rc;
}

extern "C" int dbl_sweep(dbl_ctx *ctx, int sampler, int32_t n_sweeps) {
  if (!ctx) return DBL_ERR_INVALID;
  if (ctx->async_open) { ctx->set_error("dbl_sweep with asynchronous sweeps pending: call dbl_sync first"); return DBL_ERR_STATE; }
  int rc = dbl_sweep_async(ctx, sampler, n_sweeps);
  if (rc) { ctx->async_open = false; return rc; }
  return dbl_sync(ctx);
}

// ---------------------------------------------------------------------------------------------------
// block-level entry points: one call per k-d-tree block, mirroring GibbsUpdates.updatePartition (GU:156-211)
// ---------------------------------------------------------------------------------------------------
extern "C" int dbl_block_sweep_begin(dbl_ctx *ctx, int sampler) {
  if (!ctx) return DBL_ERR_INVALID;
  if (sampler < 0 || sampler > 3) { ctx->set_error("bad sampler"); return DBL_ERR_INVALID; }
  if (!ctx->has_state) { ctx->set_error("no state"); return DBL_ERR_STATE; }
  if (ctx->world > 1) { ctx->set_error("block-level sweeps need an unsharded context"); return DBL_ERR_STATE; }
  if (ctx->in_sweep || ctx->async_open) { ctx->set_error("a sweep is already open"); return DBL_ERR_STATE; }
  CUDA_TRY(cudaSetDevice(ctx->device));
  CUDA_TRY(cudaEventRecord(ctx->ev0, ctx->stream));
  int rc = enqueue_theta(ctx);
  if (rc) return rc;
  // block membership is fixed for the whole sweep (the shuffle happens after every partition was updated, GU:144)
  CUDA_TRY(ctx->blk_frozen.alloc(ctx->E));
  CUDA_TRY(cudaMemcpyAsync(ctx->blk_frozen.p, ctx->blk.p, sizeof(int) * ctx->E, cudaMemcpyDeviceToDevice, ctx->stream));
  ctx->block_done.assign(ctx->P, 0);
  ctx->block_sampler = sampler;
  ctx->in_sweep = true;
  ctx->in_block_sweep = true;
  return DBL_OK;
}

extern "C" int dbl_update_block(dbl_ctx *ctx, int32_t block_id) {
  if (!ctx) return DBL_ERR_INVALID;
  if (!ctx->in_block_sweep) { ctx->set_error("dbl_update_block outside dbl_block_sweep_begin/end"); return DBL_ERR_STATE; }
  if (block_id < 0 || block_id >= ctx->P) { ctx->set_error("block id out of range"); return DBL_ERR_INVALID; }
  if (ctx->block_done[block_id]) { ctx->set_error("block already updated in this sweep"); return DBL_ERR_STATE; }
  CUDA_TRY(cudaSetDevice(ctx->device));
  k_mark_ent_block<<<grid_for(ctx->E, 256), 256, 0, ctx->stream>>>(ctx->E, ctx->blk_frozen.p, block_id, ctx->ent_owned.p);
  k_mark_rec_owned<<<grid_for(ctx->R, 256), 256, 0, ctx->stream>>>(ctx->R, ctx->link.p, ctx->ent_owned.p,
                                                                  ctx->rec_owned.p);
  ctx->launches += 2;
  int rc = relayout(ctx);  // tiles of this block only (everything else sorts into the dummy block)
  if (rc) return rc;
  rc = update_owned(ctx, ctx->block_sampler);
  if (rc) return rc;
  ctx->block_done[block_id] = 1;
  return DBL_OK;
}

extern "C" int dbl_block_sweep_end(dbl_ctx *ctx) {
  if (!ctx) return DBL_ERR_INVALID;
  if (!ctx->in_block_sweep) { ctx->set_error("dbl_block_sweep_end without dbl_block_sweep_begin"); return DBL_ERR_STATE; }
  for (int b = 0; b < ctx->P; ++b)
    if (!ctx->block_done[b]) { ctx->set_error("dbl_block_sweep_end: not every block was updated"); return DBL_ERR_STATE; }
  CUDA_TRY(cudaSetDevice(ctx->device));
  ctx->in_sweep = ctx->in_block_sweep = false;
  CUDA_TRY(cudaMemsetAsync(ctx->ent_owned.p, 1, ctx->E, ctx->stream));
  CUDA_TRY(cudaMemsetAsync(ctx->rec_owned.p, 1, ctx->R, ctx->stream));
  int rc = build_links_csr(ctx);
  if (rc) return rc;
  rc = refresh_summary(ctx, false);  // summary of the whole state (updateSummaryVariables, GU:219-301)
  if (rc) return rc;
  rc = adopt_local_summary(ctx);
  if (rc) return rc;
  rc = relayout(ctx);  // the shuffle: regroup by the new block ids
  if (rc) return rc;
  k_finish<<<1, 32, 0, ctx->stream>>>(ctx->ctl());
  ctx->launches += 1;
  CUDA_TRY(cudaEventRecord(ctx->ev1, ctx->stream));
  rc = snapshot(ctx);
  float ms = 0.f;
  if (cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1) == cudaSuccess) ctx->last_sweep_ms = ms;
  return rc;
}

// ---------------------------------------------------------------------------------------------------
// multi-GPU entry points: blocks are sharded over ranks; one exchange of moved clusters per sweep
// ---------------------------------------------------------------------------------------------------
static int apply_ownership(dbl_ctx *ctx) {
  k_mark_ent_owned<<<grid_for(ctx->E, 256), 256, 0, ctx->stream>>>(ctx->E, ctx->blk.p, ctx->owner.p, ctx->rank,
                                                                  ctx->ent_owned.p);
  k_mark_rec_owned<<<grid_for(ctx->R, 256), 256, 0, ctx->stream>>>(ctx->R, ctx->link.p, ctx->ent_owned.p,
                                                                  ctx->rec_owned.p);
  ctx->launches += 2;
  CUDA_TRY(cudaGetLastError());
  return DBL_OK;
}

extern "C" int dbl_set_block_owners(dbl_ctx *ctx, const int32_t *owner_of_block) {
  if (!ctx) return DBL_ERR_INVALID;
  if (!ctx->has_state) { ctx->set_error("set_block_owners needs a (replicated) state"); return DBL_ERR_STATE; }
  if (!ctx->all_owned) { ctx->set_error("set_block_owners needs the replicated state: upload / init it again first"); return DBL_ERR_STATE; }
  CUDA_TRY(cudaSetDevice(ctx->device));
  if (owner_of_block) {  // NULL = the table the context already holds on the device (the device-side LPT may have changed it)
    for (int b = 0; b < ctx->P; ++b)
      if (owner_of_block[b] < 0 || owner_of_block[b] >= ctx->world) { ctx->set_error("owner out of range"); return DBL_ERR_INVALID; }
    ctx->owner_h.assign(owner_of_block, owner_of_block + ctx->P);
    CUDA_TRY(cudaMemcpyAsync(ctx->owner.p, ctx->owner_h.data(), sizeof(int) * ctx->P, cudaMemcpyHostToDevice, ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
  }
  int rc = apply_ownership(ctx);
  if (rc) return rc;
  ctx->all_owned = (ctx->world <= 1);
  rc = build_links_csr(ctx);  // of the shard; the global summary (of the replicated state) stays
  if (rc) return rc;
  rc = relayout(ctx);
  if (rc) return rc;
  return snapshot(ctx);
}

extern "C" int dbl_block_owners(dbl_ctx *ctx, int32_t *owner_out) {
  if (!ctx || !owner_out) return DBL_ERR_INVALID;
  if (!ctx->owner.p) { ctx->set_error("no state"); return DBL_ERR_STATE; }
  CUDA_TRY(cudaSetDevice(ctx->device));
  CUDA_TRY(cudaMemcpyAsync(owner_out, ctx->owner.p, sizeof(int) * ctx->P, cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_TRY(cudaStreamSynchronize(ctx->stream));
  return DBL_OK;
}

extern "C" int dbl_set_rebalance(dbl_ctx *ctx, int32_t period, double threshold) {
  if (!ctx || period < 0 || !(threshold >= 1.0)) return DBL_ERR_INVALID;
  ctx->drop_graphs();
  ctx->rebalance_period = period;
  ctx->rebalance_threshold = threshold;
  return DBL_OK;
}

// With lazy module loading (the CUDA default) the FIRST launch of a kernel may synchronise the whole context.  Inside a
// sharded sweep that is fatal when several ranks share one device (the tests do): rank A waits in the exchange barrier
// for rank B, whose next launch waits for A's barrier kernel to finish.  So every kernel a sweep can launch is loaded
// here, before the first sharded sweep (and before any graph capture): by attribute query for our own kernels, by
// running the (idempotent) layout / index builds once for the CUB kernels they use.
static int preload_kernels(dbl_ctx *ctx) {
  cudaFuncAttributes fa;
#define DBL_LOAD(k) CUDA_TRY(cudaFuncGetAttributes(&fa, k))
  DBL_LOAD(k_theta); DBL_LOAD(k_link_heavy); DBL_LOAD(k_commit_link_keys); DBL_LOAD(k_build_tiles); DBL_LOAD(k_values<DBL_VALUES_UB_LARGE>); DBL_LOAD(k_values<8>); DBL_LOAD(k_values_log); DBL_LOAD(k_entity_post); DBL_LOAD(k_dist);
  DBL_LOAD(k_reduce_local); DBL_LOAD(k_finish); DBL_LOAD(k_move_ent); DBL_LOAD(k_move_rec); DBL_LOAD(k_publish_barrier);
  DBL_LOAD(k_unpack_ent_p2p); DBL_LOAD(k_unpack_rec_p2p); DBL_LOAD(k_reduce_peers); DBL_LOAD(k_lpt);
  DBL_LOAD(k_link_generic); DBL_LOAD(k_link_match); DBL_LOAD(k_link_pruned); DBL_LOAD(k_state_hash);
  DBL_LOAD(k_gather_ent); DBL_LOAD(k_gather_rec); DBL_LOAD(k_export_ent); DBL_LOAD(k_export_rec);
  DBL_LOAD(k_inv_keys); DBL_LOAD(k_inv_keys32); DBL_LOAD(k_inv_value_ptr32); DBL_LOAD(k_inv_segments);
#undef DBL_LOAD
  if (pcg2_kernel_fits(ctx)) {
    LinkParams lp;
    memset(&lp, 0, sizeof(lp));
    lp.hslots = ctx->hslots; lp.pack_consts = ctx->pack_consts; lp.qtile_pk = ctx->qtile_pk;
    int rc = dispatch_pcg2(ctx, 0, lp);  // grid 0 = load only
    if (rc) return rc;
  }
  int rc = build_links_csr(ctx);
  if (rc) return rc;
  ctx->inv_valid = false;
  rc = ensure_inverted_index(ctx);
  if (rc) return rc;
  rc = relayout(ctx);
  if (rc) return rc;
  CUDA_TRY(cudaStreamSynchronize(ctx->stream));
  return DBL_OK;
}

// ---- peer-to-peer communicator ------------------------------------------------------------------------------
static size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

extern "C" int dbl_comm_export(dbl_ctx *ctx, void *blob_out) {
  if (!ctx || !blob_out) return DBL_ERR_INVALID;
  if (!ctx->has_state) { ctx->set_error("dbl_comm_export needs a state (the buffers are sized by it)"); return DBL_ERR_STATE; }
  CUDA_TRY(cudaSetDevice(ctx->device));
  CUDA_TRY(cudaStreamSynchronize(ctx->stream));
  comm_close(ctx);
  ctx->drop_graphs();
  CommDev &c = ctx->comm;
  memset(&c, 0, sizeof(c));
  c.rank = ctx->rank; c.world = ctx->world; c.A = ctx->A; c.nws = ctx->nw + 1;
  c.cap_e = ctx->E; c.cap_r = ctx->R;
  c.off_cursor = 256;
  c.off_slots = 512;
  c.off_ent = align_up(c.off_slots + 2 * (size_t)c.world * c.nws * 8, 256);
  c.off_rec = align_up(c.off_ent + 2 * (size_t)c.cap_e * (c.A + 1) * 4, 256);
  const size_t bytes = align_up(c.off_rec + 2 * (size_t)c.cap_r * 3 * 4, 256);
  if (ctx->comm_bytes != bytes || !ctx->comm_buf.p) {
    CUDA_TRY(ctx->comm_buf.alloc(bytes));
    ctx->comm_bytes = bytes;
  }
  CUDA_TRY(cudaMemset(ctx->comm_buf.p, 0, 512 + 2 * (size_t)c.world * c.nws * 8));
  long long zero = 0;  // barrier epochs restart with the buffers
  CUDA_TRY(cudaMemcpy(ctx->ctl() + CTL_EPOCH, &zero, sizeof(zero), cudaMemcpyHostToDevice));
  CommBlob b;
  memset(&b, 0, sizeof(b));
  b.magic = COMM_MAGIC; b.rank = ctx->rank; b.world = ctx->world; b.device = ctx->device;
  b.pid = (int64_t)getpid();
  b.ptr = (uint64_t)(uintptr_t)ctx->comm_buf.p;
  b.bytes = bytes; b.E = ctx->E; b.R = ctx->R; b.A = ctx->A; b.nws = c.nws;
  if (ctx->world > 1 && cudaIpcGetMemHandle(&b.handle, ctx->comm_buf.p) != cudaSuccess) {
    // no IPC on this system: ranks living in this process still reach the buffer through b.ptr; a rank in another
    // process will fail in dbl_comm_import and the host layer falls back to the host-mediated exchange
    cudaGetLastError();
    memset(&b.handle, 0, sizeof(b.handle));
  }
  memcpy(blob_out, &b, sizeof(b));
  return DBL_OK;
}

extern "C" int dbl_comm_import(dbl_ctx *ctx, const void *blobs, int32_t world) {
  if (!ctx || !blobs) return DBL_ERR_INVALID;
  if (world != ctx->world) { ctx->set_error("dbl_comm_import: world size differs from the context's"); return DBL_ERR_INVALID; }
  if (!ctx->comm_buf.p) { ctx->set_error("dbl_comm_import before dbl_comm_export"); return DBL_ERR_STATE; }
  CUDA_TRY(cudaSetDevice(ctx->device));
  const CommBlob *bl = static_cast<const CommBlob *>(blobs);
  for (int r = 0; r < world; ++r) {
    CommBlob b;
    memcpy(&b, &bl[r], sizeof(b));
    if (b.magic != COMM_MAGIC || b.rank != r || b.world != world || b.E != ctx->E || b.R != ctx->R || b.A != ctx->A ||
        b.nws != ctx->comm.nws || b.bytes != ctx->comm_bytes) {
      ctx->set_error("dbl_comm_import: blob " + std::to_string(r) + " does not describe a matching rank");
      return DBL_ERR_INVALID;
    }
    if (r == ctx->rank) {
      ctx->comm.base[r] = ctx->comm_buf.p;
    } else if (b.pid == (int64_t)getpid()) {  // several ranks in one process (tests): plain pointers
      if (b.device != ctx->device) {
        cudaError_t e = cudaDeviceEnablePeerAccess(b.device, 0);
        if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) { ctx->set_error("no peer access between the devices"); return DBL_ERR_CUDA; }
        cudaGetLastError();
      }
      ctx->comm.base[r] = reinterpret_cast<unsigned char *>((uintptr_t)b.ptr);
    } else {
      void *p = nullptr;
      cudaError_t e = cudaIpcOpenMemHandle(&p, b.handle, cudaIpcMemLazyEnablePeerAccess);
      if (e != cudaSuccess) {
        ctx->set_error(std::string("cudaIpcOpenMemHandle (rank ") + std::to_string(r) + "): " + cudaGetErrorString(e));
        comm_close(ctx);
        return DBL_ERR_CUDA;
      }
      ctx->ipc_opened.push_back(p);
      ctx->comm.base[r] = static_cast<unsigned char *>(p);
    }
  }
  ctx->drop_graphs();
  if (ctx->has_state) { int rc = preload_kernels(ctx); if (rc) return rc; }
  ctx->comm_ready = true;
  return DBL_OK;
}

extern "C" int dbl_last_exchange(dbl_ctx *ctx, int64_t *ent_msgs, int64_t *rec_msgs, int64_t *replacements) {
  if (!ctx || !ctx->h_cb) return DBL_ERR_INVALID;
  if (ent_msgs) *ent_msgs = ctx->h_ctl()[CTL_MOVED_ENT];
  if (rec_msgs) *rec_msgs = ctx->h_ctl()[CTL_MOVED_REC];
  if (replacements) *replacements = ctx->h_ctl()[CTL_REPLACED];
  return DBL_OK;
}

// ---- host-mediated exchange ---------------------------------------------------------------------------------
extern "C" int dbl_sweep_begin(dbl_ctx *ctx, int sampler, int64_t *ent_counts, int64_t *rec_counts) {
  if (!ctx || !ent_counts || !rec_counts) return DBL_ERR_INVALID;
  if (sampler < 0 || sampler > 3) { ctx->set_error("bad sampler"); return DBL_ERR_INVALID; }
  if (!ctx->has_state) { ctx->set_error("no state"); return DBL_ERR_STATE; }
  if (ctx->in_sweep || ctx->async_open) { ctx->set_error("dbl_sweep_begin twice"); return DBL_ERR_STATE; }
  CUDA_TRY(cudaSetDevice(ctx->device));
  CUDA_TRY(cudaEventRecord(ctx->ev0, ctx->stream));
  int rc = enqueue_theta(ctx);
  if (rc) return rc;
  rc = update_owned(ctx, sampler);
  if (rc) return rc;
  const int W = ctx->world;
  CUDA_TRY(cudaMemsetAsync(ctx->move_cnt.p, 0, sizeof(unsigned long long) * 4 * W, ctx->stream));
  k_move_count_ent<<<grid_for(ctx->E, 256), 256, 0, ctx->stream>>>(ctx->E, ctx->blk.p, ctx->owner.p, ctx->rank,
                                                                  ctx->ent_owned.p, ctx->ent_dest.p, ctx->move_cnt.p);
  k_move_count_rec<<<grid_for(ctx->R, 256), 256, 0, ctx->stream>>>(ctx->R, ctx->link.p, ctx->rec_owned.p,
                                                                  ctx->ent_dest.p, ctx->move_cnt.p + W);
  ctx->launches += 2;
  std::vector<unsigned long long> h(2 * W);
  CUDA_TRY(cudaMemcpyAsync(h.data(), ctx->move_cnt.p, sizeof(unsigned long long) * 2 * W, cudaMemcpyDeviceToHost, ctx->stream));
  rc = snapshot(ctx);  // also the partial summary of the shard (dbl_partial_summary) and the sweep's status
  ctx->h_move_ent.assign(W, 0);
  ctx->h_move_rec.assign(W, 0);
  for (int d = 0; d < W; ++d) {
    ent_counts[d] = ctx->h_move_ent[d] = (int64_t)h[d];
    rec_counts[d] = ctx->h_move_rec[d] = (int64_t)h[W + d];
  }
  if (rc) {  // abandoned: nothing leaves this rank, but the caller still runs the collective calls of the sweep
    for (int d = 0; d < W; ++d) ent_counts[d] = rec_counts[d] = ctx->h_move_ent[d] = ctx->h_move_rec[d] = 0;
  }
  ctx->in_sweep = true;
  return rc;
}

extern "C" int dbl_exchange_pack(dbl_ctx *ctx, void *ent_buf_dev, void *rec_buf_dev) {
  if (!ctx) return DBL_ERR_INVALID;
  if (!ctx->in_sweep) { ctx->set_error("dbl_exchange_pack outside a sweep"); return DBL_ERR_STATE; }
  CUDA_TRY(cudaSetDevice(ctx->device));
  const int W = ctx->world;
  std::vector<unsigned long long> cur(2 * W);
  unsigned long long oe = 0, orc = 0;
  for (int d = 0; d < W; ++d) { cur[d] = oe; oe += ctx->h_move_ent[d]; cur[W + d] = orc; orc += ctx->h_move_rec[d]; }
  CUDA_TRY(cudaMemcpyAsync(ctx->move_cnt.p + 2 * W, cur.data(), sizeof(unsigned long long) * 2 * W, cudaMemcpyHostToDevice,
                           ctx->stream));
  if (orc > 0) {
    if (!rec_buf_dev) return DBL_ERR_INVALID;
    k_move_pack_rec<<<grid_for(ctx->R, 256), 256, 0, ctx->stream>>>(ctx->R, ctx->link.p, ctx->zmask.p, ctx->ent_dest.p,
                                                                   ctx->rec_owned.p, ctx->move_cnt.p + 3 * W,
                                                                   (int *)rec_buf_dev);
  }
  if (oe > 0) {
    if (!ent_buf_dev) return DBL_ERR_INVALID;
    k_move_pack_ent<<<grid_for(ctx->E, 256), 256, 0, ctx->stream>>>(ctx->E, ctx->A, ctx->y.p, ctx->ent_dest.p,
                                                                   ctx->ent_owned.p, ctx->move_cnt.p + 2 * W,
                                                                   (int *)ent_buf_dev);
  }
  ctx->launches += 2;
  CUDA_TRY(cudaGetLastError());
  CUDA_TRY(cudaStreamSynchronize(ctx->stream));  // the host moves the buffers with NCCL on its own stream
  return DBL_OK;
}

extern "C" int dbl_exchange_unpack(dbl_ctx *ctx, const void *ent_buf_dev, int64_t n_ent, const void *rec_buf_dev,
                                   int64_t n_rec) {
  if (!ctx || n_ent < 0 || n_rec < 0) return DBL_ERR_INVALID;
  if (!ctx->in_sweep) { ctx->set_error("dbl_exchange_unpack outside a sweep"); return DBL_ERR_STATE; }
  CUDA_TRY(cudaSetDevice(ctx->device));
  if (n_ent > 0)
    k_unpack_ent<<<grid_for(n_ent, 256), 256, 0, ctx->stream>>>(n_ent, ctx->A, (const int *)ent_buf_dev, ctx->attrs.p,
                                                                ctx->tree, ctx->y.p, ctx->entN.p, ctx->blk.p,
                                                                ctx->ent_owned.p);
  if (n_rec > 0)
    k_unpack_rec<<<grid_for(n_rec, 256), 256, 0, ctx->stream>>>(n_rec, (const int *)rec_buf_dev, ctx->link.p,
                                                                ctx->zmask.p, ctx->rec_owned.p);
  ctx->launches += 2;
  CUDA_TRY(cudaGetLastError());
  CUDA_TRY(cudaStreamSynchronize(ctx->stream));
  return DBL_OK;
}

// global_counts = the all-reduced words of dbl_partial_summary (drives the next theta draw); failed != 0: some rank
// reported an error for this sweep, so it is abandoned on every rank
extern "C" int dbl_sweep_end(dbl_ctx *ctx, const int64_t *global_counts, double global_loglik, int32_t failed) {
  if (!ctx || !global_counts) return DBL_ERR_INVALID;
  if (!ctx->in_sweep) { ctx->set_error("dbl_sweep_end without dbl_sweep_begin"); return DBL_ERR_STATE; }
  CUDA_TRY(cudaSetDevice(ctx->device));
  ctx->in_sweep = false;
  if (failed) {
    ctx->has_state = false;
    ctx->set_error("the sweep failed on a peer rank");
    return DBL_ERR_CUDA;
  }
  std::vector<long long> g(ctx->n_counts());
  for (int i = 0; i < ctx->n_counts(); ++i) g[i] = global_counts[i];
  memcpy(&g[ctx->ll_slot()], &global_loglik, sizeof(double));
  CUDA_TRY(cudaMemcpyAsync(ctx->glob(), g.data(), sizeof(long long) * ctx->n_counts(), cudaMemcpyHostToDevice, ctx->stream));
  CUDA_TRY(cudaStreamSynchronize(ctx->stream));
  int rc = relayout(ctx);
  if (rc) return rc;
  k_finish<<<1, 32, 0, ctx->stream>>>(ctx->ctl());
  ctx->launches += 1;
  CUDA_TRY(cudaEventRecord(ctx->ev1, ctx->stream));
  rc = snapshot(ctx);
  float ms = 0.f;
  if (cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1) == cudaSuccess) ctx->last_sweep_ms = ms;
  return rc;
}

// partial summary of the shard after dbl_sweep_begin / dbl_set_block_owners (host copy, no device work)
extern "C" int dbl_partial_summary(dbl_ctx *ctx, int64_t *counts, double *loglik) {
  if (!ctx || !counts || !loglik) return DBL_ERR_INVALID;
  for (int i = 0; i < ctx->n_counts(); ++i) counts[i] = ctx->h_part()[i];
  counts[ctx->ll_slot()] = 0;
  memcpy(loglik, &ctx->h_part()[ctx->ll_slot()], sizeof(double));
  return DBL_OK;
}
extern "C" int32_t dbl_summary_words(const dbl_ctx *ctx) { return ctx ? ctx->n_counts() : 0; }

extern "C" int dbl_export_owned_dev(dbl_ctx *ctx, void *y_dev, void *blk_dev, void *link_dev, void *z_dev) {
  if (!ctx || !y_dev || !blk_dev || !link_dev || !z_dev) return DBL_ERR_INVALID;
  if (!ctx->has_state) { ctx->set_error("no state"); return DBL_ERR_STATE; }
  CUDA_TRY(cudaSetDevice(ctx->device));
  k_export_ent<<<grid_for(ctx->E, 256), 256, 0, ctx->stream>>>(ctx->E, ctx->A, ctx->ent_owned.p, ctx->y.p, ctx->blk.p,
                                                              (int *)y_dev, (int *)blk_dev);
  k_export_rec<<<grid_for(ctx->R, 256), 256, 0, ctx->stream>>>(ctx->R, ctx->A, ctx->rec_owned.p, ctx->link.p,
                                                              ctx->zmask.p, (int *)link_dev, (unsigned char *)z_dev);
  ctx->launches += 2;
  CUDA_TRY(cudaGetLastError());
  CUDA_TRY(cudaStreamSynchronize(ctx->stream));
  return DBL_OK;
}

// the rows this rank owns, compacted (block-major order): ids + rows.  Host buffers sized for E / R rows.
extern "C" int dbl_download_owned(dbl_ctx *ctx, int64_t *n_ent, int32_t *ent_ids, int32_t *y, int32_t *block,
                                  int64_t *n_rec, int32_t *rec_ids, int32_t *link, uint8_t *z) {
  if (!ctx || !n_ent || !n_rec) return DBL_ERR_INVALID;
  if (!ctx->has_state) { ctx->set_error("no state"); return DBL_ERR_STATE; }
  if (ctx->world > 1 && ctx->all_owned) { ctx->set_error("dbl_download_owned before dbl_set_block_owners"); return DBL_ERR_STATE; }
  CUDA_TRY(cudaSetDevice(ctx->device));
  if (ctx->h_owned_ent < 0 || ctx->h_owned_rec < 0) { int rc = snapshot(ctx); if (rc) return rc; }
  const int64_t ne = ctx->h_owned_ent, nr = ctx->h_owned_rec;
  const int A = ctx->A;
  *n_ent = ne; *n_rec = nr;
  if (!(ent_ids && y && block) && !(rec_ids && link && z)) return DBL_OK;  // counts only
  const size_t need_i = (size_t)(ne * (A + 2) + nr * 2) + 1;
  if (ctx->gather_i.n < need_i) CUDA_TRY(ctx->gather_i.alloc(need_i));
  if (ctx->gather_b.n < (size_t)nr * A + 1) CUDA_TRY(ctx->gather_b.alloc((size_t)nr * A + 1));
  int *eids = ctx->gather_i.p, *yo = eids + ne, *bo = yo + ne * A, *rids = bo + ne, *lo = rids + nr;
  if (ne > 0 && ent_ids && y && block) {
    k_gather_ent<<<grid_for(ne, 256), 256, 0, ctx->stream>>>(ne, A, ctx->ent_sorted.p, ctx->y.p, ctx->blk.p, eids, yo, bo);
    CUDA_TRY(cudaMemcpyAsync(ent_ids, eids, sizeof(int) * ne, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(cudaMemcpyAsync(y, yo, sizeof(int) * ne * A, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(cudaMemcpyAsync(block, bo, sizeof(int) * ne, cudaMemcpyDeviceToHost, ctx->stream));
  }
  if (nr > 0 && rec_ids && link && z) {
    k_gather_rec<<<grid_for(nr, 256), 256, 0, ctx->stream>>>(nr, A, ctx->rec_sorted.p, ctx->link.p, ctx->zmask.p, rids, lo,
                                                            ctx->gather_b.p);
    CUDA_TRY(cudaMemcpyAsync(rec_ids, rids, sizeof(int) * nr, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(cudaMemcpyAsync(link, lo, sizeof(int) * nr, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(cudaMemcpyAsync(z, ctx->gather_b.p, (size_t)nr * A, cudaMemcpyDeviceToHost, ctx->stream));
  }
  ctx->launches += 2;
  CUDA_TRY(cudaGetLastError());
  CUDA_TRY(cudaStreamSynchronize(ctx->stream));
  return DBL_OK;
}

extern "C" int dbl_owned_masks(dbl_ctx *ctx, uint8_t *ent_owned, uint8_t *rec_owned) {
  if (!ctx) return DBL_ERR_INVALID;
  if (!ctx->has_state) { ctx->set_error("no state"); return DBL_ERR_STATE; }
  CUDA_TRY(cudaSetDevice(ctx->device));
  if (ent_owned) CUDA_TRY(cudaMemcpyAsync(ent_owned, ctx->ent_owned.p, ctx->E, cudaMemcpyDeviceToHost, ctx->stream));
  if (rec_owned) CUDA_TRY(cudaMemcpyAsync(rec_owned, ctx->rec_owned.p, ctx->R, cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_TRY(cudaStreamSynchronize(ctx->stream));
  return DBL_OK;
}

// fingerprint of the rows this rank owns: hash[0] entities (id, values), hash[1] records (id, link, distortion bits);
// the sums over ranks mod 2^64 identify the global state whatever the number of ranks or the placement
extern "C" int dbl_state_hash(dbl_ctx *ctx, uint64_t *hash_out) {
  if (!ctx || !hash_out) return DBL_ERR_INVALID;
  if (!ctx->has_state) { ctx->set_error("no state"); return DBL_ERR_STATE; }
  CUDA_TRY(cudaSetDevice(ctx->device));
  CUDA_TRY(cudaMemsetAsync(ctx->hash_words(), 0, 2 * sizeof(unsigned long long), ctx->stream));
  k_state_hash<<<grid_rows(std::max(ctx->E, ctx->R), 256), 256, 0, ctx->stream>>>(
      rows_masked(ctx, true), rows_masked(ctx, false), ctx->A, ctx->y.p, ctx->link.p, ctx->zmask.p, ctx->hash_words());
  ctx->launches += 1;
  unsigned long long h[2] = {0, 0};
  CUDA_TRY(cudaMemcpyAsync(h, ctx->hash_words(), sizeof(h), cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_TRY(cudaStreamSynchronize(ctx->stream));
  hash_out[0] = h[0]; hash_out[1] = h[1];
  return DBL_OK;
}

// which link kernel a sweep with this sampler launches: 0 k_link_generic, 1 k_link_match, 2 k_link_pruned,
// 3 k_link_pcg2 (+4 when the constants are byte-packed, +8 when the hash tables have the compile-time 32 slots)
extern "C" int dbl_link_kernel(const dbl_ctx *ctx, int sampler) {
  if (!ctx || sampler < 0 || sampler > 3) return DBL_ERR_INVALID;
  const int mode = ctx->link_mode;
  if (mode != 1 && sampler == DBL_PCG_II && pcg2_kernel_fits(ctx))
    return 3 + (ctx->qtile_pk ? 4 : 0) + (ctx->hslots == 32 ? 8 : 0);
  if (mode == 0 && sampler != DBL_PCG_II) return 2;
  const size_t ring = (size_t)LINK_STAGES * tile_words(ctx->A) * 4 + 128;
  if (mode != 1 && sampler != DBL_PCG_II && ring <= 160 * 1024) return 1;
  return 0;
}

extern "C" int dbl_set_link_mode(dbl_ctx *ctx, int mode) {
  if (!ctx || mode < 0 || mode > 2) return DBL_ERR_INVALID;
  ctx->drop_graphs();
  ctx->link_mode = mode;
  return DBL_OK;
}

extern "C" double dbl_last_sweep_ms(const dbl_ctx *ctx) { return ctx ? ctx->last_sweep_ms : 0.0; }

extern "C" double dbl_link_kernel_ms(dbl_ctx *ctx, int64_t *launches) {
  if (!ctx) return 0.0;
  const double ms = ctx->link_ms;
  if (launches) *launches = ctx->link_launches;
  ctx->link_ms = 0.0;
  ctx->link_launches = 0;
  return ms;
}

extern "C" int64_t dbl_phase_ms(dbl_ctx *ctx, double *out4) {
  if (!ctx || !out4) return 0;
  const int64_t n = ctx->phase_sweeps;
  for (int i = 0; i < 4; ++i) { out4[i] = ctx->phase_ms[i]; ctx->phase_ms[i] = 0.0; }
  ctx->phase_sweeps = 0;
  return n;
}

extern "C" int dbl_summary(dbl_ctx *ctx, dbl_summary_head *head, int64_t *agg_dist, int64_t *rec_dist, double *theta) {
  if (!ctx) return DBL_ERR_INVALID;
  if (!ctx->has_state) { ctx->set_error("no state"); return DBL_ERR_STATE; }
  const int A = ctx->A, F = ctx->F;
  const long long *g = ctx->h_glob();
  if (head) {
    head->iteration = ctx->iteration;
    head->num_isolates = g[ctx->iso_slot()];
    double ll;
    memcpy(&ll, &g[ctx->ll_slot()], sizeof(double));
    for (int a = 0; a < A; ++a)
      for (int f = 0; f < F; ++f) {  // GU:286-293
        const double th = ctx->h_theta[a * F + f];
        const double nd = (double)g[a * F + f];
        ll += (ctx->alpha[a] + nd - 1.0) * std::log(th) +
              (ctx->beta[a] + (double)ctx->file_sizes[f] - nd - 1.0) * std::log(1.0 - th);
      }
    head->log_likelihood = ll;
    head->pairs_scored = ctx->h_pairs;
  }
  if (agg_dist) for (int i = 0; i < A * F; ++i) agg_dist[i] = g[i];
  if (rec_dist) for (int i = 0; i <= A; ++i) rec_dist[i] = g[A * F + i];
  if (theta) std::copy(ctx->h_theta.begin(), ctx->h_theta.end(), theta);
  return DBL_OK;
}
