// cml_gibbs.cu -- collapsed Gibbs sampling (carmel --crp) over the resident derivation lattices (K8).
//
// Reference semantics (restated, not copied):
//   gibbs_base::iteration            graehl/shared/gibbs.hpp:836-877   (remove block, resample, add block)
//   gibbs_param proposal_prob/addc   graehl/shared/gibbs.hpp:154-157,203-211
//   carmel_gibbs::operator()/choose  carmel/src/gibbs.cc:348-371       (arc prob = product of chain params)
//   derivations::random_path         carmel/src/derivations.h:345-375  (backward filter, forward sample)
//   pfor::global_normalize, choose_p derivations.h:318-337 ; graehl/shared/random.ipp:111-127
// One uniform per visited non-final lattice state, in path order.  The uniforms are counter based
// (seed, sweep, block, draw) so that any block can be sampled on any GPU thread and still reproduce the
// same derivation as the sequential CPU restatement.
//
// Modes
//   sequential (exact): ONE CTA walks the blocks in corpus order; every block sees the counts that include
//     the blocks sampled before it in this sweep, exactly like the reference (latency bound by design).
//   batched: one WARP per block, all blocks sampled in parallel against the counts of the previous sweep minus
//     the block's own previous sample (a synchronous version of "remove block, resample, add block"); the count
//     deltas are applied afterwards with fp64 REDs.  Not sample-identical to the sequential sampler by
//     construction; reported as final-perplexity agreement (tests/test_gibbs_gpu.py).
#include <algorithm>
#include <cmath>

#include "cml_ctx.cuh"

namespace {

__device__ __forceinline__ double gibbs_uniform(uint64_t seed, uint32_t sweep, uint32_t block, uint32_t draw) {
  uint64_t h = mix64(seed ^ mix64(((uint64_t)sweep << 32) | block));
  h = mix64(h + draw);
  return (double)(h >> 11) * (1.0 / 9007199254740992.0);
}

struct GibbsArgs {
  const CmlExDesc* desc;
  uint32_t n_ex;
  const uint32_t* lvl_off;
  const uint32_t* out_off;
  const uint2* out_arc;        // {dst layered index, internal arc id}
  const uint32_t* arc_orig;    // internal arc id -> arc-table id
  const uint32_t* chain_off;   // arc-table id -> parameters (NULL: arc i is parameter i)
  const uint32_t* chain_param;
  const uint32_t* param_norm;  // CML_NO_GROUP: fixed probability = prior
  const double* prior;
  double* count;
  double* normsum;
  const double* arc_lnw;       // per internal arc id (batched mode / initial sample from EM weights), may be NULL
  const uint32_t* au_off;      // per internal arc id: its parameters that have a CRP normalisation group (CSR)
  const uint32_t* au_param;
  const uint2* arc_pg;         // per internal arc id: {the one adjustable parameter, its group}; x = ~0 none, ~0-1 several (use the CSR)
  double* beta;               // scratch: one double per lattice state
  const uint64_t* beta_base;
  const uint64_t* sample_base;
  const uint32_t* old_sample;  // arc-table ids of the previous sample
  const uint32_t* old_len;
  uint32_t* new_sample;
  uint32_t* new_len;
  double power;
  uint64_t seed;
  uint32_t sweep;
  int sequential;
};

__device__ __forceinline__ double param_prob(const GibbsArgs& A, uint32_t p) {
  const uint32_t g = A.param_norm[p];
  return g == CML_NO_GROUP ? A.prior[p] : A.count[p] / A.normsum[g];
}
__device__ double arc_lnprob(const GibbsArgs& A, uint32_t internal_id) {
  if (A.arc_lnw) return A.arc_lnw[internal_id];
  const uint32_t a = A.arc_orig[internal_id];
  if (!A.chain_off) return log(param_prob(A, a));
  double s = 0;
  for (uint32_t k = A.chain_off[a], e = A.chain_off[a + 1]; k < e; ++k) s += log(param_prob(A, A.chain_param[k]));
  return s;
}
__device__ void add_sample_counts(const GibbsArgs& A, const uint32_t* arcs, uint32_t n, double d, bool atomic) {
  for (uint32_t i = 0; i < n; ++i) {
    const uint32_t a = arcs[i];
    const uint32_t k0 = A.chain_off ? A.chain_off[a] : a, k1 = A.chain_off ? A.chain_off[a + 1] : a + 1;
    for (uint32_t k = k0; k < k1; ++k) {
      const uint32_t p = A.chain_off ? A.chain_param[k] : k;
      const uint32_t g = A.param_norm[p];
      if (g == CML_NO_GROUP) continue;
      if (atomic) {
        atomicAdd(&A.count[p], d);
        atomicAdd(&A.normsum[g], d);
      } else {
        A.count[p] += d;
        A.normsum[g] += d;
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------------
// One block (example) by a group of NT threads (NT = 32: a warp, batched mode; NT = blockDim: the CTA of the
// sequential mode).  Backward filter over the layered CSR in log space, then a forward sample.
//   backward, per level: phase 1 -- threads over the level's ARCS (coalesced 8-byte records, independent
//   gathers of the arc's ln probability and beta[dst]) stage v = ln w + beta[dst] in shared memory;
//   phase 2 -- threads over the level's STATES fold their contiguous run of staged values (online LSE, arcs in
//   the stored order).  Levels with more arcs than the stage are processed in chunks.
//   forward: the first warp evaluates the current state's arcs in parallel, lane 0 then replays the
//   reference's three sequential loops (sum, psum, running choice; derivations.h:318-337, random.ipp:111-127)
//   on the staged values, so the selected arc -- and the rounding that selects it -- is the sequential one.
// ---------------------------------------------------------------------------------------------------
// Batched mode, "remove the block before resampling it" (gibbs.hpp:844-859): every block is sampled against the
// previous sweep's counts MINUS its own previous sample.  The subtraction is kept per block in two small shared
// hash tables (parameter -> ln(1 - own/count), normalisation group -> -ln(1 - own/normsum)) and added to the frozen
// per-arc table entry of every arc whose adjustable parameters they touch.
const int kOwnCap = 128;  // entries per table (power of two); a block with more distinct parameters keeps the rest unadjusted
struct OwnTables {
  uint32_t* kp;
  double* vp;
  uint32_t* kg;
  double* vg;
};
__device__ __forceinline__ uint32_t own_hash(uint32_t key) { return (key * 2654435761u) >> 25; }  // 7 bits
__device__ __forceinline__ int own_find(const uint32_t* keys, uint32_t key) {
  uint32_t i = own_hash(key);
  for (int probe = 0; probe < kOwnCap; ++probe, i = (i + 1) & (kOwnCap - 1)) {
    const uint32_t k = keys[i];
    if (k == key) return (int)i;
    if (k == 0xFFFFFFFFu) return -1;
  }
  return -1;
}
__device__ __forceinline__ void own_add(uint32_t* keys, double* vals, uint32_t key, double d) {
  uint32_t i = own_hash(key);
  for (int probe = 0; probe < kOwnCap - 8; ++probe, i = (i + 1) & (kOwnCap - 1)) {  // keep a few slots free: finds terminate
    const uint32_t prev = atomicCAS(&keys[i], 0xFFFFFFFFu, key);
    if (prev == 0xFFFFFFFFu || prev == key) {
      atomicAdd(&vals[i], d);
      return;
    }
  }
}
__device__ void own_build(const GibbsArgs& A, uint32_t e, int lane, const OwnTables& T) {
  for (int i = lane; i < kOwnCap; i += 32) {
    T.kp[i] = 0xFFFFFFFFu;
    T.kg[i] = 0xFFFFFFFFu;
    T.vp[i] = 0;
    T.vg[i] = 0;
  }
  __syncwarp();
  const uint32_t* arcs = A.old_sample + A.sample_base[e];
  const uint32_t n = A.old_len[e];
  const double wt = A.desc[e].weight;
  for (uint32_t i = lane; i < n; i += 32) {
    const uint32_t a = arcs[i];
    const uint32_t k0 = A.chain_off ? A.chain_off[a] : a, k1 = A.chain_off ? A.chain_off[a + 1] : a + 1;
    for (uint32_t k = k0; k < k1; ++k) {
      const uint32_t p = A.chain_off ? A.chain_param[k] : k;
      const uint32_t g = A.param_norm[p];
      if (g == CML_NO_GROUP) continue;
      own_add(T.kp, T.vp, p, wt);
      own_add(T.kg, T.vg, g, wt);
    }
  }
  __syncwarp();
  for (int i = lane; i < kOwnCap; i += 32) {
    if (T.kp[i] != 0xFFFFFFFFu) {
      const double r = 1. - T.vp[i] / A.count[T.kp[i]];
      T.vp[i] = r > 0 ? log(r) : -CUDART_INF;
    }
    if (T.kg[i] != 0xFFFFFFFFu) {
      const double r = 1. - T.vg[i] / A.normsum[T.kg[i]];
      T.vg[i] = r > 0 ? -log(r) : 0.;
    }
  }
  __syncwarp();
}
__device__ __forceinline__ double own_correction(const GibbsArgs& A, const OwnTables* T, uint32_t internal_id) {
  if (!T) return 0.;
  double c = 0;
  const uint2 pg = __ldg(&A.arc_pg[internal_id]);  // the common cases in one load: no / exactly one adjustable parameter
  if (pg.x == 0xFFFFFFFFu) return 0.;
  if (pg.x != 0xFFFFFFFEu) {
    const int ig = own_find(T->kg, pg.y);
    if (ig < 0) return 0.;
    c = T->vg[ig];
    const int ip = own_find(T->kp, pg.x);
    return ip >= 0 ? c + T->vp[ip] : c;
  }
  for (uint32_t k = A.au_off[internal_id], k1 = A.au_off[internal_id + 1]; k < k1; ++k) {
    const uint32_t p = A.au_param[k];
    const int ig = own_find(T->kg, A.param_norm[p]);
    if (ig < 0) continue;
    c += T->vg[ig];
    const int ip = own_find(T->kp, p);
    if (ip >= 0) c += T->vp[ip];
  }
  return c;
}

template <int NT>
__device__ __forceinline__ void gsync() {
  if (NT == 32)
    __syncwarp();
  else
    __syncthreads();
}
template <int NT>
__device__ void sample_block(const GibbsArgs& A, uint32_t e, int tid, double* __restrict__ stage, uint32_t cap,
                             const OwnTables* own = nullptr) {
  const CmlExDesc d = A.desc[e];
  const uint32_t* __restrict__ lvl = A.lvl_off + d.lvl_base;
  const uint32_t* __restrict__ ooff = A.out_off + d.row_base;
  const uint2* __restrict__ oarc = A.out_arc + d.arc_base;
  double* be = A.beta + A.beta_base[e];
  const double NI = -CUDART_INF;
  const int nl = (int)d.n_levels;
  const int nt = NT == 32 ? 32 : (int)blockDim.x;
  for (int L = nl - 1; L >= 0; --L) {
    const uint32_t s0 = lvl[L], s1 = lvl[L + 1];
    for (uint32_t st0 = s0; st0 < s1; st0 += nt) {  // a tile of nt states and the arcs that leave them
      const uint32_t st1 = min(st0 + (uint32_t)nt, s1);
      const uint32_t t0 = ooff[st0], t1 = ooff[st1];
      const uint32_t s = st0 + tid;
      uint32_t r0 = 0, r1 = 0;
      double m = NI, acc = 0;
      if (s < st1) {
        r0 = ooff[s];
        r1 = ooff[s + 1];
        if (s == d.fin) {
          m = 0;
          acc = 1;
        }
      }
      for (uint32_t c0 = t0; c0 < t1; c0 += cap) {
        const uint32_t c1 = min(c0 + cap, t1);
#pragma unroll 4
        for (uint32_t k = c0 + tid; k < c1; k += nt) {
          const uint2 r = oarc[k];
          stage[k - c0] = arc_lnprob(A, r.y) + own_correction(A, own, r.y) + be[r.x];
        }
        gsync<NT>();
        for (uint32_t k = max(r0, c0), ke = min(r1, c1); k < ke; ++k) {
          const double v = stage[k - c0];
          if (v > m) {
            acc = acc * exp(m - v) + 1.;
            m = v;
          } else if (v > NI)
            acc += exp(v - m);
        }
        gsync<NT>();
      }
      if (s < st1) be[s] = (m > NI) ? m + log(acc) : NI;
    }
    gsync<NT>();
  }
  if (tid < 32) {  // forward sample by the first warp
    const int lane = tid;
    uint32_t* out = A.new_sample + A.sample_base[e];
    uint32_t n = 0, s = 0, draw = 0;  // the start state has layered index 0
    while (s != d.fin) {
      const uint32_t k0 = ooff[s], k1 = ooff[s + 1];
      if (k0 == k1) break;  // cannot happen on a pruned lattice
      const uint32_t deg = k1 - k0;
      uint32_t pick = k1 - 1;
      if (deg <= cap) {
        // global_normalize: nw = (w*beta)^power ; p = nw / sum -- values staged once, loops replayed by lane 0
        for (uint32_t j = lane; j < deg; j += 32) {
          const uint2 r = oarc[k0 + j];
          stage[j] = A.power * (arc_lnprob(A, r.y) + own_correction(A, own, r.y) + be[r.x]);
        }
        __syncwarp();
        if (lane == 0) {
          double m = NI;
          for (uint32_t j = 0; j < deg; ++j) m = fmax(m, stage[j]);
          double sum = 0;
          for (uint32_t j = 0; j < deg; ++j) {
            const double v = stage[j];
            const double ex = v > NI ? exp(v - m) : 0.;
            stage[j] = ex;
            sum += ex;
          }
          double psum = 0;
          for (uint32_t j = 0; j < deg; ++j) {
            const double pj = sum > 0 ? stage[j] / sum : 0.;
            stage[j] = pj;
            psum += pj;
          }
          double choice = psum * gibbs_uniform(A.seed, A.sweep, d.ex_index, draw);
          for (uint32_t j = 0; j < deg; ++j) {
            choice -= stage[j];
            if (choice < 0) {
              pick = k0 + j;
              break;
            }
          }
        }
      } else if (lane == 0) {  // very wide state: recompute per pass (no staging)
        double m = NI;
        for (uint32_t k = k0; k < k1; ++k) {
          const uint2 r = oarc[k];
          m = fmax(m, A.power * (arc_lnprob(A, r.y) + own_correction(A, own, r.y) + be[r.x]));
        }
        double sum = 0;
        for (uint32_t k = k0; k < k1; ++k) {
          const uint2 r = oarc[k];
          const double v = A.power * (arc_lnprob(A, r.y) + own_correction(A, own, r.y) + be[r.x]);
          if (v > NI) sum += exp(v - m);
        }
        double psum = 0;
        for (uint32_t k = k0; k < k1; ++k) {
          const uint2 r = oarc[k];
          const double v = A.power * (arc_lnprob(A, r.y) + own_correction(A, own, r.y) + be[r.x]);
          psum += (v > NI && sum > 0) ? exp(v - m) / sum : 0.;
        }
        double choice = psum * gibbs_uniform(A.seed, A.sweep, d.ex_index, draw);
        for (uint32_t k = k0; k < k1; ++k) {
          const uint2 r = oarc[k];
          const double v = A.power * (arc_lnprob(A, r.y) + own_correction(A, own, r.y) + be[r.x]);
          choice -= (v > NI && sum > 0) ? exp(v - m) / sum : 0.;
          if (choice < 0) {
            pick = k;
            break;
          }
        }
      }
      ++draw;
      pick = __shfl_sync(0xffffffffu, pick, 0);
      const uint2 pr = oarc[pick];
      if (lane == 0) out[n] = A.arc_orig[pr.y];
      ++n;
      s = pr.x;
      __syncwarp();
    }
    if (lane == 0) A.new_len[e] = n;
  }
  gsync<NT>();
}

const int kGibbsStage = 384;       // staged arc values per warp (batched mode): 3 KB (+3 KB of own-sample tables => 37 warps/SM)
const int kGibbsWarps = 4;
const int kGibbsSeqThreads = 1024;
const int kGibbsSeqStage = 4096;   // sequential mode: one CTA, 32 KB stage

// batched mode: one warp per block, every block against the frozen per-arc table of this sweep
__global__ void __launch_bounds__(kGibbsWarps * 32) k_gibbs_batched(GibbsArgs A) {
  __shared__ double stage_all[kGibbsWarps * kGibbsStage];
  __shared__ double own_v[kGibbsWarps * 2 * kOwnCap];
  __shared__ uint32_t own_k[kGibbsWarps * 2 * kOwnCap];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  double* stage = stage_all + warp * kGibbsStage;
  OwnTables T;
  T.kp = own_k + warp * 2 * kOwnCap;
  T.kg = T.kp + kOwnCap;
  T.vp = own_v + warp * 2 * kOwnCap;
  T.vg = T.vp + kOwnCap;
  for (uint32_t e = blockIdx.x * kGibbsWarps + warp; e < A.n_ex; e += gridDim.x * kGibbsWarps) {
    const bool excl = A.au_off != nullptr && A.old_len[e] != 0;
    if (excl) own_build(A, e, lane, T);
    sample_block<32>(A, e, lane, stage, kGibbsStage, excl ? &T : nullptr);
  }
}

// sequential (exact) mode: one CTA walks the blocks in corpus order; counts updated in place between blocks and the
// per-arc ln-probability table rebuilt from them (all threads) before every block
__global__ void __launch_bounds__(kGibbsSeqThreads) k_gibbs_sequential(GibbsArgs A, double* __restrict__ tbl, uint32_t n_tbl) {
  __shared__ double stage[kGibbsSeqStage];
  GibbsArgs B = A;
  B.arc_lnw = tbl;
  for (uint32_t e = 0; e < A.n_ex; ++e) {
    const double wt = A.desc[e].weight;
    if (threadIdx.x == 0) add_sample_counts(A, A.old_sample + A.sample_base[e], A.old_len[e], -wt, false);
    __syncthreads();
    if (!A.arc_lnw) {
      for (uint32_t a = threadIdx.x; a < n_tbl; a += blockDim.x) tbl[a] = arc_lnprob(A, a);
      __syncthreads();
    }
    sample_block<kGibbsSeqThreads>(A.arc_lnw ? A : B, e, (int)threadIdx.x, stage, kGibbsSeqStage);
    if (threadIdx.x == 0) add_sample_counts(A, A.new_sample + A.sample_base[e], A.new_len[e], wt, false);
    __syncthreads();
  }
}


// --expectation (gibbs.cc:311-316, derivations.h:381-398 collect_counts_gibbs): a block's "sample" is every arc of its
// lattice with its posterior under the current proposal probabilities (incremental EM over the CRP counts).  One CTA
// walks the blocks in corpus order: the block's previous posteriors leave the counts, the lattice arcs get their
// proposal weights from the counts, forward / backward in log space (online log-sum-exp in stored arc order), the new
// posteriors enter the counts.  post[] holds one double per lattice arc (out-arc order), old and new generation.
struct ExpectArgs {
  const uint32_t* in_off;
  const uint2* in_arc;      // {src layered index, internal arc id}, destination-major
  double* alpha;            // scratch: one double per lattice state (same bases as beta)
  const double* old_post;
  double* new_post;
  double* blk_lnp;          // [n_ex] ln P(block) = sum over all derivations
};
__global__ void __launch_bounds__(kGibbsSeqThreads) k_gibbs_expectation(GibbsArgs A, ExpectArgs X) {
  const double NI = -CUDART_INF;
  const int tid = (int)threadIdx.x, nt = (int)blockDim.x;
  for (uint32_t e = 0; e < A.n_ex; ++e) {
    const CmlExDesc d = A.desc[e];
    const uint32_t* __restrict__ lvl = A.lvl_off + d.lvl_base;
    const uint32_t* __restrict__ ooff = A.out_off + d.row_base;
    const uint32_t* __restrict__ ioff = X.in_off + d.row_base;
    const uint2* __restrict__ oarc = A.out_arc + d.arc_base;
    const uint2* __restrict__ iarc = X.in_arc + d.arc_base;
    const double* __restrict__ po = X.old_post + d.arc_base;
    double* __restrict__ pn = X.new_post + d.arc_base;
    double* be = A.beta + A.beta_base[e];
    double* al = X.alpha + A.beta_base[e];
    const uint32_t n_arcs = ooff[d.n_states];
    const double wt = d.weight;
    auto for_params = [&](uint32_t internal, double dlt) {  // addc with block_delta weights (gibbs.hpp:779-786)
      const uint32_t a = A.arc_orig[internal];
      const uint32_t k0 = A.chain_off ? A.chain_off[a] : a, k1 = A.chain_off ? A.chain_off[a + 1] : a + 1;
      for (uint32_t k = k0; k < k1; ++k) {
        const uint32_t p = A.chain_off ? A.chain_param[k] : k;
        const uint32_t g = A.param_norm[p];
        if (g == CML_NO_GROUP) continue;
        atomicAdd(&A.count[p], dlt);
        atomicAdd(&A.normsum[g], dlt);
      }
    };
    // (1) the block's previous posteriors leave the counts
    for (uint32_t k = tid; k < n_arcs; k += nt) {
      const double v = po[k];
      if (v != 0.) for_params(oarc[k].y, -wt * v);
    }
    __syncthreads();
    // (2) proposal weight of every lattice arc from the counts as they are now (fixed for the whole block)
    for (uint32_t k = tid; k < n_arcs; k += nt) pn[k] = arc_lnprob(A, oarc[k].y);
    __syncthreads();
    // (3) backward, levels descending: a thread per state, arcs in stored order
    for (int L = (int)d.n_levels - 1; L >= 0; --L) {
      for (uint32_t s = lvl[L] + tid; s < lvl[L + 1]; s += nt) {
        double m = NI, acc = 0;
        if (s == d.fin) {
          m = 0;
          acc = 1;
        }
        for (uint32_t k = ooff[s], ke = ooff[s + 1]; k < ke; ++k) {
          const double v = pn[k] + be[oarc[k].x];
          if (v > m) {
            acc = acc * exp(m - v) + 1.;
            m = v;
          } else if (v > NI)
            acc += exp(v - m);
        }
        be[s] = (m > NI) ? m + log(acc) : NI;
      }
      __syncthreads();
    }
    // (4) forward, levels ascending, over the incoming arcs; the weight of in-arc j is looked up through its arc id
    for (uint32_t L = 0; L < d.n_levels; ++L) {
      for (uint32_t s = lvl[L] + tid; s < lvl[L + 1]; s += nt) {
        double m = NI, acc = 0;
        if (s == 0) {
          m = 0;
          acc = 1;
        }
        for (uint32_t k = ioff[s], ke = ioff[s + 1]; k < ke; ++k) {
          const uint2 r = iarc[k];
          const double v = arc_lnprob(A, r.y) + al[r.x];
          if (v > m) {
            acc = acc * exp(m - v) + 1.;
            m = v;
          } else if (v > NI)
            acc += exp(v - m);
        }
        al[s] = (m > NI) ? m + log(acc) : NI;
      }
      __syncthreads();
    }
    const double lnP = al[d.fin];
    if (tid == 0) X.blk_lnp[e] = lnP;
    // (5) posteriors (count updates only after every thread has read the counts it needs: steps 2 and 4 are done)
    for (uint32_t s = tid; s < d.n_states; s += nt) {
      const double a_s = al[s];
      for (uint32_t k = ooff[s], ke = ooff[s + 1]; k < ke; ++k) {
        const double v = pn[k] + a_s + be[oarc[k].x] - lnP;
        pn[k] = (lnP > NI && v > NI) ? exp(v) : 0.;
      }
    }
    __syncthreads();
    for (uint32_t k = tid; k < n_arcs; k += nt) {
      const double v = pn[k];
      if (v != 0.) for_params(oarc[k].y, wt * v);
    }
    __syncthreads();
  }
}

// ---------------------------------------------------------------------------------------------------
// Dense-state batched sampler (cml_gibbs_attach_dense): position-synchronous lattices are never walked.
// One warp per block, lane = WFST state.  Backward filter in scaled linear space: beta_t[i] = sum_j W[o_t][j][i] *
// c_t[j] * beta_{t+1}[j] with W the per-sweep dense table of arc probabilities (stored [symbol][destination][source]
// so a lane's reads are coalesced) and c_t[j] the block's own-sample correction of the (j, o_t) parameters; the vector
// is renormalised by a power of two every step (only ratios matter to the sampler).  Forward: from state s, lane j
// holds (W[o_t][j][s] c_t[j] beta_{t+1}[j])^power, one warp scan turns the uniform draw into the successor state.
// ---------------------------------------------------------------------------------------------------
struct DenseGibbs {
  uint32_t S, V, start, fin;
  const uint32_t* arc;   // [(o*S+j)*32+i] internal arc id or 0xFFFFFFFF
  const uint32_t* rep;   // [o*S+j] internal id of an arc whose adjustable parameters are those of (j,o), or 0xFFFFFFFF
  const uint64_t* seq_off;
  const uint16_t* sym;
  const double* W;       // [(o*S+j)*32+i] linear probability (0 where there is no arc)
  double* beta;          // rows of 32
};
__global__ void k_gibbs_dense_table(uint32_t n, const uint32_t* __restrict__ arc, const double* __restrict__ arc_lnw,
                                    double* __restrict__ W) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint32_t a = arc[i];
  W[i] = a == 0xFFFFFFFFu ? 0. : exp(arc_lnw[a]);
}
__global__ void __launch_bounds__(kGibbsWarps * 32) k_gibbs_dense(GibbsArgs A, DenseGibbs G) {
  __shared__ __align__(16) double stage_all[kGibbsWarps * 32];
  __shared__ double own_v[kGibbsWarps * 2 * kOwnCap];
  __shared__ uint32_t own_k[kGibbsWarps * 2 * kOwnCap];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  double* stage = stage_all + warp * 32;
  OwnTables T;
  T.kp = own_k + warp * 2 * kOwnCap;
  T.kg = T.kp + kOwnCap;
  T.vp = own_v + warp * 2 * kOwnCap;
  T.vg = T.vp + kOwnCap;
  const uint32_t S = G.S;
  for (uint32_t e = blockIdx.x * kGibbsWarps + warp; e < A.n_ex; e += gridDim.x * kGibbsWarps) {
    const bool excl = A.au_off != nullptr && A.old_len[e] != 0;
    if (excl) own_build(A, e, lane, T);
    const uint64_t base = G.seq_off[e];
    const uint32_t n = (uint32_t)(G.seq_off[e + 1] - base);
    const uint16_t* __restrict__ sy = G.sym + base;
    double* __restrict__ be = G.beta + (base + e) * 32 + lane;
    auto corr = [&](uint32_t o) -> double {  // multiplicative own-sample correction of the (lane, o) parameters
      if (!excl || (uint32_t)lane >= S) return 1.;
      const uint32_t r = __ldg(&G.rep[o * S + lane]);
      return r == 0xFFFFFFFFu ? 1. : exp(own_correction(A, &T, r));
    };
    // ---- backward filter
    double b = (lane == (int)G.fin) ? 1. : 0.;
    for (uint32_t t = n; t-- > 0;) {
      const uint32_t o = sy[t];
      const double cb = b * corr(o);  // what the forward pass needs of position t+1: correction x beta
      stage[lane] = cb;
      be[(size_t)(t + 1) * 32] = cb;
      __syncwarp();
      const double* __restrict__ Wo = G.W + (size_t)o * S * 32 + lane;
      double acc0 = 0, acc1 = 0, acc2 = 0, acc3 = 0;
      uint32_t j = 0;
      for (; j + 3 < S; j += 4) {
        const double2 s01 = *reinterpret_cast<const double2*>(stage + j);
        const double2 s23 = *reinterpret_cast<const double2*>(stage + j + 2);
        acc0 = fma(__ldg(Wo + (size_t)j * 32), s01.x, acc0);
        acc1 = fma(__ldg(Wo + (size_t)(j + 1) * 32), s01.y, acc1);
        acc2 = fma(__ldg(Wo + (size_t)(j + 2) * 32), s23.x, acc2);
        acc3 = fma(__ldg(Wo + (size_t)(j + 3) * 32), s23.y, acc3);
      }
      for (; j < S; ++j) acc0 = fma(__ldg(Wo + (size_t)j * 32), stage[j], acc0);
      acc0 += acc2;
      acc1 += acc3;
      b = acc0 + acc1;
      const int mx = __reduce_max_sync(0xffffffffu, __double2hiint(b));
      if (mx > 0) {
        const int ex = min(max(((mx >> 20) & 0x7ff) - 1023, -1022), 1022);
        b *= __hiloint2double((1023 - ex) << 20, 0);
      }
      __syncwarp();
    }
    // ---- forward sample
    uint32_t* out = A.new_sample + A.sample_base[e];
    uint32_t s = G.start;
    const uint32_t ex_index = A.desc[e].ex_index;
    for (uint32_t t = 0; t < n; ++t) {
      const uint32_t o = sy[t];
      double v = 0;
      if ((uint32_t)lane < S) v = __ldg(G.W + ((size_t)o * S + lane) * 32 + s) * be[(size_t)(t + 1) * 32];
      if (A.power != 1. && v > 0) v = exp(A.power * log(v));
      double m = v;
      for (int k = 16; k; k >>= 1) m = fmax(m, __shfl_xor_sync(0xffffffffu, m, k));
      double p = m > 0 ? v / m : 0.;
      double sum = p;
      for (int k = 16; k; k >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, k);
      p = sum > 0 ? p / sum : 0.;
      double cum = p;  // inclusive scan over the lanes (destination states in ascending order)
      for (int k = 1; k < 32; k <<= 1) {
        const double up = __shfl_up_sync(0xffffffffu, cum, k);
        if (lane >= k) cum += up;
      }
      const double psum = __shfl_sync(0xffffffffu, cum, 31);
      const double choice = psum * gibbs_uniform(A.seed, A.sweep, ex_index, t);
      const unsigned hit = __ballot_sync(0xffffffffu, p > 0 && choice - cum < 0);
      const unsigned any = __ballot_sync(0xffffffffu, p > 0);
      uint32_t pick = hit ? (uint32_t)(__ffs(hit) - 1) : (any ? (uint32_t)(31 - __clz(any)) : 0u);
      if (lane == 0) {
        const uint32_t a = __ldg(&G.arc[((size_t)o * S + pick) * 32 + s]);
        out[t] = a == 0xFFFFFFFFu ? 0u : A.arc_orig[a];
      }
      s = pick;
    }
    if (lane == 0) A.new_len[e] = n;
    __syncwarp();
  }
}

// batched mode: apply (new - old) sample counts of every block
__global__ void k_gibbs_apply(GibbsArgs A) {
  const uint32_t e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= A.n_ex) return;
  const double wt = A.desc[e].weight;
  add_sample_counts(A, A.old_sample + A.sample_base[e], A.old_len[e], -wt, true);
  add_sample_counts(A, A.new_sample + A.sample_base[e], A.new_len[e], wt, true);
}

// sharded batched sweeps (SURVEY 8(e)): a rank applies its blocks' (new - old) sample counts to a zeroed DELTA table
// [n_params | n_norms], the tables are summed over the ranks (one all-reduce per sweep) and added to the replicated
// counts, so every rank samples the next sweep against the same global counts
__global__ void k_gibbs_add_delta(uint32_t n_params, uint32_t n_norms, const double* __restrict__ delta, double* __restrict__ count,
                                  double* __restrict__ normsum) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n_params)
    count[i] += delta[i];
  else if (i < n_params + n_norms)
    normsum[i - n_params] += delta[i];
}

__global__ void k_gibbs_lnprob(uint32_t n_params, const uint32_t* __restrict__ param_norm, const double* __restrict__ prior,
                               const double* __restrict__ count, const double* __restrict__ normsum,
                               double* __restrict__ lnp) {
  const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= n_params) return;
  const uint32_t g = param_norm[p];
  const double v = g == CML_NO_GROUP ? prior[p] : count[p] / normsum[g];
  lnp[p] = v > 0 ? log(v) : -CUDART_INF;
}

__global__ void k_gibbs_accumulate(uint32_t n_params, const double* __restrict__ count, double* __restrict__ cum, double dt) {
  const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p < n_params) cum[p] += dt * count[p];
}

}  // namespace

extern "C" int cml_gibbs_init(cml_ctx* ctx, const cml_gibbs_model* g) {
  if (!ctx || !g) return CML_ERR_ARG;
  CML_REQUIRE(ctx->have_model, CML_ERR_STATE, "cml_set_model first");
  CML_REQUIRE(g->n_params == ctx->n_params && g->param_norm && g->param_prior, CML_ERR_ARG, "gibbs model does not match the model");
  CML_REQUIRE(ctx->batches.size() == 1 && ctx->batches[0]->ell_ex == 0, CML_ERR_STATE,
              "Gibbs sampling needs the lattices in ONE batch in the layered-CSR layout (log space or CML_OPT_NO_ELL)");
  CML_REQUIRE(ctx->batches[0]->cyc_ex == 0, CML_ERR_CYCLE,
              "Gibbs sampling over a lattice with a cycle is not built (the backward filter has no level order)");
  cudaSetDevice(ctx->device);
  Batch& bt = *ctx->batches[0];
  cudaStream_t s = ctx->stream;
  std::vector<double> normsum(std::max<uint32_t>(1, g->n_norms), 0.), count(g->n_params);
  for (uint32_t p = 0; p < g->n_params; ++p) {
    const uint32_t n = g->param_norm[p];
    CML_REQUIRE(n == CML_NO_GROUP || n < g->n_norms, CML_ERR_ARG, "param_norm out of range");
    count[p] = g->param_prior[p];
    if (n != CML_NO_GROUP) normsum[n] += g->param_prior[p];  // restore_p0 (gibbs.hpp:618-623)
  }
  ctx->g_norms = g->n_norms;
  CML_CUDA(ctx->g_param_norm.upload(g->param_norm, g->n_params, s));
  CML_CUDA(ctx->g_prior.upload(g->param_prior, g->n_params, s));
  CML_CUDA(ctx->g_count.upload(count.data(), count.size(), s));
  CML_CUDA(ctx->g_normsum.upload(normsum.data(), normsum.size(), s));
  CML_CUDA(ctx->g_cum.alloc(g->n_params));
  CML_CUDA(cudaMemsetAsync(ctx->g_cum.p, 0, g->n_params * sizeof(double), s));
  CML_CUDA(ctx->g_lnp.alloc(g->n_params));
  std::vector<uint32_t> orig((size_t)ctx->n_arcs + 1);
  for (uint32_t a = 0; a <= ctx->n_arcs; ++a) orig[ctx->h_perm[a]] = a;
  CML_CUDA(ctx->g_arc_orig.upload(orig.data(), orig.size(), s));
  {  // per internal arc: the parameters of its chain that have a CRP group (what removing a block can change)
    std::vector<uint32_t> coff, cpar;
    if (!ctx->trivial) {
      coff.resize((size_t)ctx->n_arcs + 1);
      CML_CUDA(cudaMemcpyAsync(coff.data(), ctx->chain_off.p, coff.size() * sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
      CML_CUDA(cudaStreamSynchronize(s));
      cpar.resize(coff[ctx->n_arcs]);
      if (!cpar.empty()) CML_CUDA(cudaMemcpyAsync(cpar.data(), ctx->chain_param.p, cpar.size() * sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
      CML_CUDA(cudaStreamSynchronize(s));
    }
    std::vector<uint32_t> au_off((size_t)ctx->n_arcs + 2, 0), au_param;
    for (uint32_t i = 0; i <= ctx->n_arcs; ++i) {  // i = internal id (n_arcs = the padding arc: empty)
      if (i < ctx->n_arcs) {
        const uint32_t a = orig[i];
        const uint32_t k0 = ctx->trivial ? a : coff[a], k1 = ctx->trivial ? a + 1 : coff[a + 1];
        for (uint32_t k = k0; k < k1; ++k) {
          const uint32_t p = ctx->trivial ? k : cpar[k];
          if (g->param_norm[p] != CML_NO_GROUP) au_param.push_back(p);
        }
      }
      au_off[i + 1] = (uint32_t)au_param.size();
    }
    std::vector<uint2> pg((size_t)ctx->n_arcs + 1);
    for (uint32_t i = 0; i <= ctx->n_arcs; ++i) {
      const uint32_t n = au_off[i + 1] - au_off[i];
      if (n == 0)
        pg[i] = make_uint2(0xFFFFFFFFu, 0u);
      else if (n == 1)
        pg[i] = make_uint2(au_param[au_off[i]], g->param_norm[au_param[au_off[i]]]);
      else
        pg[i] = make_uint2(0xFFFFFFFEu, 0u);
    }
    CML_CUDA(ctx->g_arc_pg.upload(pg.data(), pg.size(), s));
    CML_CUDA(ctx->g_au_off.upload(au_off.data(), au_off.size(), s));
    CML_CUDA(ctx->g_au_param.upload(au_param.data(), au_param.size(), s));
  }
  // per-example bases: sample slots (n_levels each) and beta scratch (n_states each)
  std::vector<uint64_t> sbase(bt.n_ex + 1, 0), bbase(bt.n_ex + 1, 0);
  for (uint64_t e = 0; e < bt.n_ex; ++e) {
    sbase[e + 1] = sbase[e] + bt.h_nlevels[e];
    bbase[e + 1] = bbase[e] + (bt.h_state_base[e + 1] - bt.h_state_base[e]);
  }
  ctx->h_sample_base = sbase;
  ctx->g_sample_cap = sbase[bt.n_ex];
  CML_CUDA(ctx->g_sample_base.upload(sbase.data(), sbase.size(), s));
  CML_CUDA(ctx->g_beta_base.upload(bbase.data(), bbase.size(), s));
  CML_CUDA(ctx->g_beta.alloc(std::max<uint64_t>(1, bbase[bt.n_ex])));
  for (int i = 0; i < 2; ++i) {
    CML_CUDA(ctx->g_sample[i].alloc(std::max<uint64_t>(1, ctx->g_sample_cap)));
    CML_CUDA(ctx->g_sample_len[i].alloc(bt.n_ex));
    CML_CUDA(cudaMemsetAsync(ctx->g_sample_len[i].p, 0, bt.n_ex * sizeof(uint32_t), s));
  }
  CML_CUDA(cudaStreamSynchronize(s));
  ctx->g_cur = 0;
  ctx->have_gibbs = true;
  return CML_OK;
}

extern "C" int cml_gibbs_sweep(cml_ctx* ctx, const cml_gibbs_sweep_opts* o) {
  if (!ctx || !o) return CML_ERR_ARG;
  CML_REQUIRE(ctx->have_gibbs, CML_ERR_STATE, "cml_gibbs_init first");
  cudaSetDevice(ctx->device);
  Batch& bt = *ctx->batches[0];
  cudaStream_t s = ctx->stream;
  GibbsArgs A;
  A.desc = bt.desc.p;
  A.n_ex = (uint32_t)bt.n_ex;
  A.lvl_off = bt.lvl_off.p;
  A.out_off = bt.out_off.p;
  A.out_arc = bt.out_arc.p;
  A.arc_orig = ctx->g_arc_orig.p;
  A.chain_off = ctx->trivial ? nullptr : ctx->chain_off.p;
  A.chain_param = ctx->chain_param.p;
  A.param_norm = ctx->g_param_norm.p;
  A.prior = ctx->g_prior.p;
  A.count = ctx->g_count.p;
  A.normsum = ctx->g_normsum.p;
  A.arc_lnw = nullptr;
  A.au_off = o->init_from_params ? nullptr : ctx->g_au_off.p;  // no own-block removal when sampling from fixed EM weights
  A.au_param = ctx->g_au_param.p;
  A.arc_pg = ctx->g_arc_pg.p;
  A.beta = ctx->g_beta.p;
  A.beta_base = ctx->g_beta_base.p;
  A.sample_base = ctx->g_sample_base.p;
  A.old_sample = ctx->g_sample[ctx->g_cur].p;
  A.old_len = ctx->g_sample_len[ctx->g_cur].p;
  A.new_sample = ctx->g_sample[ctx->g_cur ^ 1].p;
  A.new_len = ctx->g_sample_len[ctx->g_cur ^ 1].p;
  A.power = o->power;
  A.seed = o->seed;
  A.sweep = o->sweep;
  A.sequential = o->mode == CML_GIBBS_SEQUENTIAL;
  const bool table = (o->init_from_params || !A.sequential) && o->mode != CML_GIBBS_EXPECTATION;
  if (table) {  // per-arc ln probabilities as a table: from the EM weights, or from the frozen counts
    const double* lnp = ctx->ln_w.p;
    if (!o->init_from_params) {
      k_gibbs_lnprob<<<cdiv(ctx->n_params, 256), 256, 0, s>>>(ctx->n_params, ctx->g_param_norm.p, ctx->g_prior.p,
                                                            ctx->g_count.p, ctx->g_normsum.p, ctx->g_lnp.p);
      ++ctx->launches;
      lnp = ctx->g_lnp.p;
    } else
      CML_REQUIRE(ctx->have_params, CML_ERR_STATE, "init_from_params needs cml_set_params");
    CML_REQUIRE(ctx->precision == 64 && ctx->space == CML_SPACE_LOG, CML_ERR_STATE,
                "Gibbs sampling runs in fp64 log space (create the context with precision 64, CML_SPACE_LOG)");
    if (const int rc = cml_arc_weights_f64(ctx, lnp)) return rc;
    A.arc_lnw = (const double*)ctx->arc_w_real.p;
  }
  // batched modes: the sweep's count update, summed over the ranks when the context has a communicator
  auto apply_batched = [&](const GibbsArgs& B) -> int {
    if (!ctx->comm || ctx->comm_size <= 1) {
      k_gibbs_apply<<<cdiv(B.n_ex, 128), 128, 0, s>>>(B);
      ++ctx->launches;
      return CML_OK;
    }
    const uint32_t n_norms = (uint32_t)ctx->g_normsum.n;
    const size_t nd = (size_t)ctx->n_params + n_norms;
    if (ctx->g_delta.n < nd) CML_CUDA(ctx->g_delta.alloc(nd));
    CML_CUDA(cudaMemsetAsync(ctx->g_delta.p, 0, nd * sizeof(double), s));
    GibbsArgs D = B;
    D.count = ctx->g_delta.p;
    D.normsum = ctx->g_delta.p + ctx->n_params;
    if (B.n_ex) k_gibbs_apply<<<cdiv(B.n_ex, 128), 128, 0, s>>>(D);
    const int rc = cml_allreduce_buffer(ctx, ctx->g_delta.p, nd);
    if (rc) return rc;
    k_gibbs_add_delta<<<cdiv(nd, 256), 256, 0, s>>>(ctx->n_params, n_norms, ctx->g_delta.p, ctx->g_count.p, ctx->g_normsum.p);
    ctx->launches += 2;
    return CML_OK;
  };
  if (o->mode == CML_GIBBS_EXPECTATION) {
    CML_REQUIRE(!o->init_from_params, CML_ERR_ARG, "--expectation has no separate initial distribution (gibbs.cc:311-313)");
    const size_t na = std::max<uint64_t>(1, bt.n_arcs), ns = std::max<uint64_t>(1, bt.n_states);
    if (ctx->g_post[0].n < na) {
      for (int k = 0; k < 2; ++k) {
        CML_CUDA(ctx->g_post[k].alloc(na));
        CML_CUDA(cudaMemsetAsync(ctx->g_post[k].p, 0, na * sizeof(double), s));
      }
      CML_CUDA(ctx->g_alpha.alloc(ns));
      CML_CUDA(ctx->g_blk_lnp.alloc(std::max<uint64_t>(1, bt.n_ex)));
    }
    A.arc_lnw = nullptr;  // proposal weights straight from the counts (they change between blocks)
    ExpectArgs X;
    X.in_off = bt.in_off.p;
    X.in_arc = bt.in_arc.p;
    X.alpha = ctx->g_alpha.p;
    X.old_post = ctx->g_post[ctx->g_cur].p;
    X.new_post = ctx->g_post[ctx->g_cur ^ 1].p;
    X.blk_lnp = ctx->g_blk_lnp.p;
    k_gibbs_expectation<<<1, kGibbsSeqThreads, 0, s>>>(A, X);
    ++ctx->launches;
  } else if (A.sequential) {
    if (ctx->g_tbl.n < (size_t)ctx->n_arcs + 1) CML_CUDA(ctx->g_tbl.alloc((size_t)ctx->n_arcs + 1));
    k_gibbs_sequential<<<1, kGibbsSeqThreads, 0, s>>>(A, ctx->g_tbl.p, ctx->n_arcs);
    ++ctx->launches;
  } else if (ctx->gd_attached) {
    DenseGibbs G;
    G.S = ctx->gd_S;
    G.V = ctx->gd_V;
    G.start = ctx->gd_start;
    G.fin = ctx->gd_fin;
    G.arc = ctx->gd_arc.p;
    G.rep = ctx->gd_rep.p;
    G.seq_off = ctx->gd_seq_off.p;
    G.sym = ctx->gd_sym.p;
    G.W = ctx->gd_W.p;
    G.beta = ctx->gd_beta.p;
    const uint32_t nt = ctx->gd_V * ctx->gd_S * 32;
    k_gibbs_dense_table<<<cdiv(nt, 256), 256, 0, s>>>(nt, ctx->gd_arc.p, A.arc_lnw, ctx->gd_W.p);
    k_gibbs_dense<<<std::max(1u, std::min<unsigned>(cdiv(A.n_ex, kGibbsWarps), (unsigned)ctx->sm_count * 16u)), kGibbsWarps * 32, 0, s>>>(A, G);
    ctx->launches += 2;
    const int rc = apply_batched(A);
    if (rc) return rc;
  } else {
    k_gibbs_batched<<<std::max(1u, std::min<unsigned>(cdiv(A.n_ex, kGibbsWarps), (unsigned)ctx->sm_count * 16u)), kGibbsWarps * 32, 0, s>>>(A);
    ++ctx->launches;
    const int rc = apply_batched(A);
    if (rc) return rc;
  }
  if (o->accumulate_dt != 0.) {
    k_gibbs_accumulate<<<cdiv(ctx->n_params, 256), 256, 0, s>>>(ctx->n_params, ctx->g_count.p, ctx->g_cum.p, o->accumulate_dt);
    ++ctx->launches;
  }
  CML_CUDA(cudaGetLastError());
  CML_CUDA(cudaStreamSynchronize(s));
  ctx->g_cur ^= 1;
  return CML_OK;
}


// --expectation: ln P(block) (sum over all derivations) of every block in the last sweep
extern "C" int cml_gibbs_get_block_logprob(cml_ctx* ctx, double* ln_p, uint64_t n) {
  if (!ctx || !ln_p) return CML_ERR_ARG;
  CML_REQUIRE(ctx->have_gibbs && ctx->g_blk_lnp.p && n <= ctx->g_blk_lnp.n, CML_ERR_STATE, "no --expectation sweep has run");
  cudaSetDevice(ctx->device);
  CML_CUDA(cudaMemcpyAsync(ln_p, ctx->g_blk_lnp.p, n * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
  CML_CUDA(cudaStreamSynchronize(ctx->stream));
  return CML_OK;
}

extern "C" int cml_gibbs_attach_dense(cml_ctx* ctx, const cml_dense_view* v, const cml_sequence_batch* b) {
  if (!ctx || !v || !b) return CML_ERR_ARG;
  CML_REQUIRE(ctx->have_gibbs, CML_ERR_STATE, "cml_gibbs_init first");
  CML_REQUIRE(v->arc_src && v->arc_dst && v->arc_sym && b->seq_off, CML_ERR_ARG, "null array");
  Batch& bt = *ctx->batches[0];
  CML_REQUIRE(b->n_seq == bt.n_ex, CML_ERR_ARG, "one sequence per resident lattice, in the same order");
  const uint32_t S = v->n_states, V = v->n_symbols, nA = ctx->n_arcs;
  if (S > 32 || V == 0 || V > 65535) {
    ctx->err = "dense-state sampler needs n_states <= 32";
    return CML_ERR_NOT_DENSE;
  }
  CML_REQUIRE(v->start < S && v->final_state < S, CML_ERR_ARG, "start / final state out of range");
  for (uint64_t e = 0; e < b->n_seq; ++e) {
    const uint64_t n = b->seq_off[e + 1] - b->seq_off[e];
    if (n + 1 != bt.h_nlevels[e]) {
      ctx->err = "a lattice is not position-synchronous (levels != symbols + 1)";
      return CML_ERR_NOT_DENSE;
    }
  }
  const uint64_t n_pos = b->seq_off[b->n_seq];
  for (uint64_t i = 0; i < n_pos; ++i) CML_REQUIRE(b->sym[i] < V, CML_ERR_ARG, "sequence symbol out of range");
  cudaSetDevice(ctx->device);
  cudaStream_t s = ctx->stream;
  // per-arc adjustable (CRP) parameters, by internal id
  std::vector<uint32_t> au_off((size_t)nA + 2), au_param;
  CML_CUDA(cudaMemcpyAsync(au_off.data(), ctx->g_au_off.p, au_off.size() * sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
  CML_CUDA(cudaStreamSynchronize(s));
  au_param.resize(au_off[nA + 1]);
  if (!au_param.empty())
    CML_CUDA(cudaMemcpyAsync(au_param.data(), ctx->g_au_param.p, au_param.size() * sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
  CML_CUDA(cudaStreamSynchronize(s));
  std::vector<uint32_t> arc((size_t)V * S * 32, 0xFFFFFFFFu), rep((size_t)V * S, 0xFFFFFFFFu);
  for (uint32_t a = 0; a < nA; ++a) {
    const uint32_t i = v->arc_src[a], j = v->arc_dst[a], o = v->arc_sym[a];
    if (i >= S || j >= S || o >= V) {
      ctx->err = "epsilon arcs / out-of-range arc triples: no dense-state sampler";
      return CML_ERR_NOT_DENSE;
    }
    uint32_t& slot = arc[((size_t)o * S + j) * 32 + i];
    if (slot != 0xFFFFFFFFu) {
      ctx->err = "parallel arcs with the same (source, destination, symbol)";
      return CML_ERR_NOT_DENSE;
    }
    const uint32_t ia = ctx->h_perm[a];
    slot = ia;
    uint32_t& r = rep[(size_t)o * S + j];
    if (r == 0xFFFFFFFFu)
      r = ia;
    else {  // the adjustable parameters must be a function of (destination, symbol)
      const uint32_t n0 = au_off[r + 1] - au_off[r], n1 = au_off[ia + 1] - au_off[ia];
      bool same = n0 == n1;
      for (uint32_t k = 0; k < n0 && same; ++k) same = au_param[au_off[r] + k] == au_param[au_off[ia] + k];
      if (!same) {
        ctx->err = "an arc's CRP parameters depend on its source state: no dense-state sampler";
        return CML_ERR_NOT_DENSE;
      }
    }
  }
  std::vector<uint16_t> sym16(std::max<uint64_t>(1, n_pos));
  for (uint64_t i = 0; i < n_pos; ++i) sym16[i] = (uint16_t)b->sym[i];
  CML_CUDA(ctx->gd_arc.upload(arc.data(), arc.size(), s));
  CML_CUDA(ctx->gd_rep.upload(rep.data(), rep.size(), s));
  CML_CUDA(ctx->gd_seq_off.upload(b->seq_off, b->n_seq + 1, s));
  CML_CUDA(ctx->gd_sym.upload(sym16.data(), sym16.size(), s));
  CML_CUDA(ctx->gd_W.alloc(arc.size()));
  CML_CUDA(ctx->gd_beta.alloc((size_t)(n_pos + b->n_seq) * 32));
  CML_CUDA(cudaStreamSynchronize(s));
  ctx->gd_S = S;
  ctx->gd_V = V;
  ctx->gd_start = v->start;
  ctx->gd_fin = v->final_state;
  ctx->gd_attached = true;
  return CML_OK;
}

extern "C" int cml_gibbs_get_samples(cml_ctx* ctx, uint32_t* path_len, uint32_t* path_arcs, uint64_t cap) {
  if (!ctx || !path_len) return CML_ERR_ARG;
  CML_REQUIRE(ctx->have_gibbs, CML_ERR_STATE, "cml_gibbs_init first");
  cudaSetDevice(ctx->device);
  Batch& bt = *ctx->batches[0];
  CML_CUDA(cudaMemcpyAsync(path_len, ctx->g_sample_len[ctx->g_cur].p, bt.n_ex * sizeof(uint32_t), cudaMemcpyDeviceToHost,
                           ctx->stream));
  if (path_arcs) {
    CML_REQUIRE(cap >= ctx->g_sample_cap, CML_ERR_ARG, "path_arcs too small (need the total number of lattice levels)");
    CML_CUDA(cudaMemcpyAsync(path_arcs, ctx->g_sample[ctx->g_cur].p, ctx->g_sample_cap * sizeof(uint32_t),
                             cudaMemcpyDeviceToHost, ctx->stream));
  }
  CML_CUDA(cudaStreamSynchronize(ctx->stream));
  return CML_OK;
}

extern "C" uint64_t cml_gibbs_sample_capacity(cml_ctx* ctx) { return ctx ? ctx->g_sample_cap : 0; }

extern "C" int cml_gibbs_get_state(cml_ctx* ctx, double* count, double* cum, double* normsum) {
  if (!ctx) return CML_ERR_ARG;
  CML_REQUIRE(ctx->have_gibbs, CML_ERR_STATE, "cml_gibbs_init first");
  cudaSetDevice(ctx->device);
  if (count) CML_CUDA(cudaMemcpyAsync(count, ctx->g_count.p, ctx->n_params * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
  if (cum) CML_CUDA(cudaMemcpyAsync(cum, ctx->g_cum.p, ctx->n_params * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
  if (normsum)
    CML_CUDA(cudaMemcpyAsync(normsum, ctx->g_normsum.p, ctx->g_norms * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
  CML_CUDA(cudaStreamSynchronize(ctx->stream));
  return CML_OK;
}
