// cml_build.cu -- device-side construction of the per-example derivation lattices (SURVEY.md section 8(f)-1).
//
// Reference: derivations::compute / derive / add_arcs / prune (carmel/src/derivations.h:479-513,572-629,640-704) and the
// uncached path's per-iteration rebuild (cached_derivs.h:77-95).  Output contract (bit for bit, checked by the byte-compare
// tests of the lattice dump): states (i, s, o) numbered in DFS pre-order from (0,0,0); at every state the label classes are
// tried in the order (eps:eps), (eps:out[o]), (in[i]:eps), (in[i]:out[o]) and within a class the WFST arcs in arc-table
// order; an arc is kept unless its destination is already known dead when it is examined; a state's stored arc list is the
// reverse of the order its arcs were kept; dead states are removed and the survivors renumbered in place.
//
// Design.  The DFS order is the contract, so an example is walked by ONE thread with an explicit stack -- the parallelism
// is over examples (a 1M-sentence corpus keeps every SM busy; the walk is pointer chasing in per-worker scratch, L2/HBM
// latency bound, hidden by tens of thousands of resident workers).  Workers are persistent threads that pull examples from
// an atomic counter; each owns a scratch region (open-addressing map (i,s,o) -> id with generation stamps, dead flags, DFS
// stack, kept-arc list, renumbering) sized for the round's capacity.  Pass 1 walks every example and records its sizes
// (examples whose walk overflows the round's capacity are retried in a later round with 4x the capacity and fewer workers);
// exact CSR offsets are prefix sums; pass 2 walks the kept examples again and writes rows and arcs at their final places.
// Nothing here touches the oracle or a CPU fallback: the host-side builder (host/trellis.cpp) stays as the product's
// default for small corpora and as the second implementation the tests compare with.
#include <algorithm>
#include <chrono>
#include <cstdlib>
#include <cstring>
#include <numeric>

#include "cml_ctx.cuh"

namespace {

struct BIo {
  const uint32_t* state_off;    // [Q+1] per WFST state: range in keys / range_begin
  const uint64_t* keys;         // sorted (in << 32 | out) per state
  const uint32_t* range_begin;  // per key: begin in ids (end = next begin)
  const uint32_t* ids;          // arc-table ids, grouped by (state, label pair), each group in arc-table order
  const uint32_t* dest;         // [n_arcs] destination state per arc-table id
  uint32_t final_state;
};
struct BCorpus {
  const uint64_t* in_off;
  const uint32_t* in_sym;
  const uint64_t* out_off;
  const uint32_t* out_sym;
};
struct __align__(16) BSlot {
  uint32_t io, s, id, gen;
};
struct __align__(16) BFrame {
  uint32_t id, io, s, phase_dead;  // phase in bits 0..2, dead in bit 8
  uint32_t cur, end, pending, pad;
};
struct BKept {
  uint32_t src, dst, id;
};
enum { B_OK = 0, B_DROPPED = 1, B_OVERFLOW = 2, B_TOOLONG = 3 };
struct BArgs {
  BIo io;
  BCorpus c;
  const uint32_t* todo;  // example numbers of this launch
  uint32_t n_todo;
  uint32_t C, K, mask;   // capacities: states (= stack depth), kept arcs; map slots - 1
  BSlot* map;
  uint8_t* dead;
  BFrame* stack;
  BKept* kept;
  uint32_t* renum;
  uint32_t* cnt;
  unsigned long long* next;     // work counter
  // pass 1 outputs (indexed by example number)
  uint8_t* status;
  uint32_t* n_states;           // live states
  uint32_t* n_arcs;             // final arcs
  uint32_t* fin;
  uint32_t* peak;               // [3] max over examples: states before pruning, kept arcs before pruning, stack depth
  unsigned long long* pre_arcs; // arcs examined
  // pass 2
  int fill;
  const uint64_t* row_base;     // [example] first entry of its arc_off row block
  const uint64_t* arc_base;
  uint32_t* out_off;
  uint32_t* out_dst;
  uint32_t* out_id;
};

__device__ __forceinline__ uint32_t b_hash(uint32_t io, uint32_t s) {
  uint32_t h = io * 0x9E3779B1u ^ (s + 0x7F4A7C15u) * 0x85EBCA6Bu;
  h ^= h >> 15;
  h *= 0xC2B2AE35u;
  return h ^ (h >> 13);
}

__global__ void __launch_bounds__(128) k_build_trellis(BArgs A) {
  const uint32_t w = blockIdx.x * blockDim.x + threadIdx.x;
  BSlot* __restrict__ map = A.map + (size_t)w * (A.mask + 1);
  uint8_t* __restrict__ dead = A.dead + (size_t)w * A.C;
  BFrame* __restrict__ stack = A.stack + (size_t)w * A.C;
  BKept* __restrict__ kept = A.kept + (size_t)w * A.K;
  uint32_t* __restrict__ renum = A.renum + (size_t)w * A.C;
  uint32_t* __restrict__ cnt = A.cnt + (size_t)w * (A.C + 1);
  uint32_t gen = 0;  // the scratch is zeroed before the launch: stamp 0 = empty
  for (;;) {
    const unsigned long long t = atomicAdd(A.next, 1ull);
    if (t >= A.n_todo) break;
    const uint32_t e = A.todo[t];
    const uint64_t i0 = A.c.in_off[e], o0 = A.c.out_off[e];
    const uint32_t nin = (uint32_t)(A.c.in_off[e + 1] - i0), nout = (uint32_t)(A.c.out_off[e + 1] - o0);
    if (nin > 65534u || nout > 65534u) {
      A.status[e] = B_TOOLONG;
      continue;
    }
    const uint32_t* __restrict__ in = A.c.in_sym + i0;
    const uint32_t* __restrict__ out = A.c.out_sym + o0;
    const uint32_t goal_io = (nin << 16) | nout, goal_s = A.io.final_state;
    ++gen;
    uint32_t n_states = 0, n_kept = 0, sp = 0, sp_max = 0;
    unsigned long long pre = 0;
    bool overflow = false;
    // map: find (io, s) or insert it with id = n_states
    auto find_or_insert = [&](uint32_t io, uint32_t s, bool& inserted) -> uint32_t {
      uint32_t h = b_hash(io, s) & A.mask;
      for (;;) {
        const BSlot sl = map[h];
        if (sl.gen != gen) {
          map[h] = BSlot{io, s, n_states, gen};
          inserted = true;
          return n_states;
        }
        if (sl.io == io && sl.s == s) {
          inserted = false;
          return sl.id;
        }
        h = (h + 1) & A.mask;
      }
    };
    BFrame f;
    {
      bool ins;
      find_or_insert(0u, 0u, ins);
      f = BFrame{0u, 0u, 0u, (goal_io == 0u && goal_s == 0u) ? 0u : 0x100u, 0u, 0u, 0u, 0u};
      dead[0] = 0;
      n_states = 1;
      sp = sp_max = 1;
    }
    while (sp) {
      if (f.cur == f.end) {
        const uint32_t ph = f.phase_dead & 7u;
        if (ph == 4u) {  // every label class done: the state is finished
          const uint32_t done = f.id, done_dead = f.phase_dead >> 8;
          dead[done] = (uint8_t)done_dead;
          if (--sp == 0) break;
          f = stack[sp - 1];  // the parent was waiting for this destination (add_arcs, derivations.h:691-701)
          if (!done_dead) {
            if (n_kept < A.K) kept[n_kept] = BKept{f.id, done, f.pending};
            else overflow = true;
            ++n_kept;
            f.phase_dead &= 7u;
          }
          continue;
        }
        f.phase_dead += 1u;  // open label class ph (derivations.h:656-670)
        const uint32_t i = f.io >> 16, o = f.io & 0xFFFFu;
        const bool useI = i < nin, useO = o < nout;
        uint32_t lin = 0, lout = 0;  // 0 = *e*
        bool active = true;
        if (ph == 1u) {
          active = useO;
          if (active) lout = out[o];
        } else if (ph == 2u) {
          active = useI;
          if (active) lin = in[i];
        } else if (ph == 3u) {
          active = useI && useO;
          if (active) {
            lin = in[i];
            lout = out[o];
          }
        }
        f.cur = f.end = 0;
        if (active) {  // arcs of WFST state f.s with this label pair (wfst_io_index, derivations.h:142-155)
          const uint64_t key = ((uint64_t)lin << 32) | lout;
          uint32_t lo = A.io.state_off[f.s], hi = A.io.state_off[f.s + 1];
          while (lo < hi) {
            const uint32_t mid = (lo + hi) >> 1;
            if (A.io.keys[mid] < key) lo = mid + 1;
            else hi = mid;
          }
          if (lo < A.io.state_off[f.s + 1] && A.io.keys[lo] == key) {
            f.cur = A.io.range_begin[lo];
            f.end = A.io.range_begin[lo + 1];
          }
        }
        continue;
      }
      // examine the next arc of the open class
      const uint32_t id = A.io.ids[f.cur++];
      ++pre;
      const uint32_t ph = (f.phase_dead & 7u) - 1u;
      const uint32_t nio = f.io + ((ph & 2u) ? 0x10000u : 0u) + (ph & 1u);
      const uint32_t ds = A.io.dest[id];
      if (n_states >= A.C) {  // (the map is kept at most half full: C <= (mask + 1) / 2)
        overflow = true;
        break;
      }
      bool ins;
      const uint32_t dst = find_or_insert(nio, ds, ins);
      if (ins) {
        f.pending = id;
        stack[sp - 1] = f;
        f = BFrame{n_states, nio, ds, (nio == goal_io && ds == goal_s) ? 0u : 0x100u, 0u, 0u, 0u, 0u};
        dead[n_states] = 0;
        ++n_states;
        ++sp;  // (sp <= n_states <= C)
        sp_max = max(sp_max, sp);
      } else if (!dead[dst]) {  // includes states still on the stack (their flag is 0 until they are finished)
        if (n_kept < A.K) kept[n_kept] = BKept{f.id, dst, id};
        else overflow = true;
        ++n_kept;
        f.phase_dead &= 7u;
      }
    }
    if (!A.fill) {
      atomicMax(A.peak + 0, n_states);
      atomicMax(A.peak + 1, n_kept);
      atomicMax(A.peak + 2, sp_max);
    }
    if (overflow) {
      A.status[e] = B_OVERFLOW;
      continue;
    }
    // the goal state
    uint32_t fin = 0xFFFFFFFFu;
    {
      uint32_t h = b_hash(goal_io, goal_s) & A.mask;
      for (;;) {
        const BSlot sl = map[h];
        if (sl.gen != gen) break;
        if (sl.io == goal_io && sl.s == goal_s) {
          fin = sl.id;
          break;
        }
        h = (h + 1) & A.mask;
      }
    }
    if (fin == 0xFFFFFFFFu || dead[fin] || dead[0]) {
      A.status[e] = B_DROPPED;
      if (!A.fill) atomicAdd(A.pre_arcs, pre);
      continue;
    }
    // prune: drop dead states keeping the order, drop arcs into them (derivations.h:612-628)
    uint32_t n_live = 0;
    for (uint32_t s = 0; s < n_states; ++s) renum[s] = dead[s] ? 0xFFFFFFFFu : n_live++;
    for (uint32_t s = 0; s <= n_live; ++s) cnt[s] = 0;
    for (uint32_t k = 0; k < n_kept; ++k) {
      const BKept a = kept[k];
      if (renum[a.src] != 0xFFFFFFFFu && renum[a.dst] != 0xFFFFFFFFu) ++cnt[renum[a.src] + 1];
    }
    for (uint32_t s = 0; s < n_live; ++s) cnt[s + 1] += cnt[s];
    if (!A.fill) {
      A.status[e] = B_OK;
      A.n_states[e] = n_live;
      A.n_arcs[e] = cnt[n_live];
      A.fin[e] = renum[fin];
      atomicAdd(A.pre_arcs, pre);
      continue;
    }
    uint32_t* __restrict__ off = A.out_off + A.row_base[e];
    uint32_t* __restrict__ adst = A.out_dst + A.arc_base[e];
    uint32_t* __restrict__ aid = A.out_id + A.arc_base[e];
    for (uint32_t s = 0; s <= n_live; ++s) off[s] = cnt[s];
    // stored list order = reverse keep order: every row is filled from its end
    for (uint32_t s = 0; s < n_live; ++s) cnt[s] = cnt[s + 1];
    for (uint32_t k = 0; k < n_kept; ++k) {
      const BKept a = kept[k];
      const uint32_t rs = renum[a.src], rd = renum[a.dst];
      if (rs == 0xFFFFFFFFu || rd == 0xFFFFFFFFu) continue;
      const uint32_t pos = --cnt[rs];
      adst[pos] = rd;
      aid[pos] = a.id;
    }
  }
}

// ---- lattices of one given string, the other tape free (carmel_b200.h, cml_build_free_trellises) ---------------------
// One warp per string over a cell grid (t, q), t in [0, |s|], q a machine state; cell (t, q) of string e is
// cell_base[e] + t * Q + q in the three scratch arrays.  Pass 0 (count): forward reachability (fw), co-reachability of
// the reachable cells (kept), then the state ids in (t, eps-level, q) order and the sizes.  Pass 1 (fill): the same
// order again, each kept state's row offset and its kept arcs (eps group and s[t] group merged back into arc-table
// order) written at the string's place in the chunk's output.
constexpr int kFreeWarps = 4;  // warps per block

struct FArgs {
  const uint32_t* key_off;    // [Q + 1] per state: its range in keys
  const uint32_t* keys;       // per state, ascending: the given-tape symbols its arcs carry (0 = *e* first)
  const uint32_t* grp;        // per key: begin in ids (end = next entry)
  const uint32_t* ids;        // arc-table ids grouped by (state, given symbol), each group in arc-table order
  const uint32_t* dest;       // [n_arcs]
  const uint32_t* order;      // [Q] states sorted by (eps-level, state)
  const uint32_t* lvl_off;    // [L + 1] eps-level l is order[lvl_off[l] .. lvl_off[l + 1])
  uint32_t Q, L, final_state;
  const uint64_t* s_off;      // [n + 1]
  const uint32_t* sym;
  uint64_t e0;                // first string of the chunk
  uint32_t n_list;            // strings of the chunk
  const uint64_t* cell_base;  // [n] first cell of each string (relative to its chunk)
  uint8_t* fw;
  uint8_t* kept;
  uint32_t* id;
  uint32_t* n_st;             // [n] kept states (0: no derivation)
  uint32_t* n_arc;            // [n] kept arcs
  int fill;
  const uint64_t* row_base;   // [n] first arc_off entry of the string in the chunk's output (fill)
  const uint64_t* arc_base;   // [n] first arc (fill)
  uint32_t* out_off;
  uint32_t* out_dst;
  uint32_t* out_id;
};

// [begin, end) in ids of the arcs of state q whose given-tape label is `symbol`
__device__ __forceinline__ uint2 f_group(const uint32_t* __restrict__ key_off, const uint32_t* __restrict__ keys,
                                         const uint32_t* __restrict__ grp, uint32_t q, uint32_t symbol) {
  uint32_t lo = key_off[q], hi = key_off[q + 1];
  const uint32_t end = hi;
  while (lo < hi) {
    const uint32_t mid = (lo + hi) >> 1;
    if (keys[mid] < symbol) lo = mid + 1;
    else hi = mid;
  }
  if (lo < end && keys[lo] == symbol) return make_uint2(grp[lo], grp[lo + 1]);
  return make_uint2(0, 0);
}

__global__ void k_build_free(FArgs A) {
  const uint32_t lane = threadIdx.x & 31;
  const uint32_t Q = A.Q, L = A.L;
  for (uint32_t w = blockIdx.x * kFreeWarps + threadIdx.x / 32; w < A.n_list; w += gridDim.x * kFreeWarps) {
    const uint64_t e = A.e0 + w;
    const uint32_t* __restrict__ s = A.sym + A.s_off[e];
    const uint32_t n = (uint32_t)(A.s_off[e + 1] - A.s_off[e]);
    const uint64_t cb = A.cell_base[e];
    uint8_t* __restrict__ fw = A.fw + cb;
    uint8_t* __restrict__ kept = A.kept + cb;
    uint32_t* __restrict__ id = A.id + cb;
    const uint32_t *key_off = A.key_off, *keys = A.keys, *grp = A.grp;
    // the arcs of q leaving position t: the *e* group (same position), the s[t] group (next position)
    auto eps_group = [=](uint32_t q) { return f_group(key_off, keys, grp, q, 0u); };
    auto sym_group = [=](uint32_t q, uint32_t t) {
      return (t < n && s[t] != 0u) ? f_group(key_off, keys, grp, q, s[t]) : make_uint2(0, 0);
    };
    if (!A.fill) {
      // forward: reachability from (0, 0); the cells are zero on entry
      if (lane == 0) fw[0] = 1;
      __syncwarp();
      for (uint32_t t = 0; t <= n; ++t) {
        const uint64_t row = (uint64_t)t * Q;
        for (uint32_t l = 0; l < L; ++l) {
          for (uint32_t j = A.lvl_off[l] + lane; j < A.lvl_off[l + 1]; j += 32) {
            const uint32_t q = A.order[j];
            if (!fw[row + q]) continue;
            const uint2 ge = eps_group(q), gs = sym_group(q, t);
            for (uint32_t k = ge.x; k < ge.y; ++k) fw[row + A.dest[A.ids[k]]] = 1;  // a later eps-level of this position
            for (uint32_t k = gs.x; k < gs.y; ++k) fw[row + Q + A.dest[A.ids[k]]] = 1;
          }
          __syncwarp();
        }
      }
      // backward: a reachable cell is kept when it is the goal or an arc leads to a kept cell
      for (uint32_t t = n + 1; t-- > 0;) {
        const uint64_t row = (uint64_t)t * Q;
        for (uint32_t l = L; l-- > 0;) {
          for (uint32_t j = A.lvl_off[l] + lane; j < A.lvl_off[l + 1]; j += 32) {
            const uint32_t q = A.order[j];
            uint8_t k = 0;
            if (fw[row + q]) {
              k = (t == n && q == A.final_state);
              const uint2 ge = eps_group(q), gs = sym_group(q, t);
              for (uint32_t a = ge.x; a < ge.y && !k; ++a) k = kept[row + A.dest[A.ids[a]]];
              for (uint32_t a = gs.x; a < gs.y && !k; ++a) k = kept[row + Q + A.dest[A.ids[a]]];
            }
            kept[row + q] = k;
          }
          __syncwarp();
        }
      }
    }
    if (!kept[0]) {  // (0, 0) does not reach the goal: no derivation
      if (!A.fill && lane == 0) A.n_st[e] = A.n_arc[e] = 0;
      continue;
    }
    // numbering in (t, eps-level, q) order; arcs counted (pass 0) or written (pass 1) in the same order
    uint32_t* __restrict__ off = A.fill ? A.out_off + A.row_base[e] : nullptr;
    uint32_t* __restrict__ odst = A.fill ? A.out_dst + A.arc_base[e] : nullptr;
    uint32_t* __restrict__ oid = A.fill ? A.out_id + A.arc_base[e] : nullptr;
    uint32_t next_id = 0, next_arc = 0;
    for (uint32_t t = 0; t <= n; ++t) {
      const uint64_t row = (uint64_t)t * Q;
      for (uint32_t j0 = 0; j0 < Q; j0 += 32) {
        const uint32_t j = j0 + lane;
        const uint32_t q = j < Q ? A.order[j] : 0u;
        const bool k = j < Q && kept[row + q];
        uint2 ge = make_uint2(0, 0), gs = make_uint2(0, 0);
        uint32_t cnt = 0;
        if (k) {
          ge = eps_group(q);
          gs = sym_group(q, t);
          for (uint32_t a = ge.x; a < ge.y; ++a) cnt += kept[row + A.dest[A.ids[a]]];
          for (uint32_t a = gs.x; a < gs.y; ++a) cnt += kept[row + Q + A.dest[A.ids[a]]];
        }
        const unsigned bal = __ballot_sync(0xFFFFFFFFu, k);
        uint32_t incl = cnt;  // inclusive warp scan of the arc counts
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
          const uint32_t v = __shfl_up_sync(0xFFFFFFFFu, incl, o);
          if ((int)lane >= o) incl += v;
        }
        if (k) {
          const uint32_t my_id = next_id + __popc(bal & ((1u << lane) - 1u));
          if (!A.fill) {
            id[row + q] = my_id;
          } else {  // row offset, then the eps group and the s[t] group merged back into arc-table order
            uint32_t p = next_arc + incl - cnt;
            off[my_id] = p;
            uint32_t a = ge.x, b = gs.x;
            while (a < ge.y || b < gs.y) {
              const bool take_e = b >= gs.y || (a < ge.y && A.ids[a] < A.ids[b]);
              const uint32_t arc = take_e ? A.ids[a++] : A.ids[b++];
              const uint64_t dc = (take_e ? row : row + Q) + A.dest[arc];
              if (!kept[dc]) continue;
              odst[p] = id[dc];
              oid[p] = arc;
              ++p;
            }
          }
        }
        next_id += __popc(bal);
        next_arc += __shfl_sync(0xFFFFFFFFu, incl, 31);
      }
    }
    if (lane == 0) {
      if (A.fill)
        off[next_id] = next_arc;
      else {
        A.n_st[e] = next_id;
        A.n_arc[e] = next_arc;
      }
    }
  }
}

struct BuiltOwner {
  std::vector<uint32_t> ex_states, ex_fin, arc_off, arc_dst, arc_id, kept_example, dropped;
  std::vector<double> ex_weight;
  cml_built_trellises pub;
};

template <typename T>
struct ScopedDev {  // cudaMalloc'ed scratch, released on scope exit
  T* p = nullptr;
  cudaError_t alloc(size_t n) { return cudaMalloc((void**)&p, std::max<size_t>(1, n) * sizeof(T)); }
  ~ScopedDev() {
    if (p) cudaFree(p);
  }
};

}  // namespace

extern "C" int cml_build_trellises(cml_ctx* ctx, const cml_wfst_view* x, const cml_corpus_view* c, cml_built_trellises** out) {
  if (!ctx || !x || !c || !out) return CML_ERR_ARG;
  *out = nullptr;
  CML_REQUIRE(x->n_states >= 1 && x->state_arc_off && (x->n_arcs == 0 || (x->arc_in && x->arc_out && x->arc_dest)), CML_ERR_ARG,
              "cml_build_trellises: incomplete transducer view");
  CML_REQUIRE(x->final_state < x->n_states, CML_ERR_ARG, "cml_build_trellises: final state out of range");
  CML_REQUIRE(c->n_ex == 0 || (c->in_off && c->out_off), CML_ERR_ARG, "cml_build_trellises: incomplete corpus view");
  CML_REQUIRE(c->n_ex < 0xFFFFFFFFull, CML_ERR_ARG, "cml_build_trellises: too many examples");
  const auto t_start = std::chrono::steady_clock::now();
  CML_CUDA(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  const uint32_t Q = x->n_states;
  const uint64_t n_arcs = x->n_arcs;
  const uint64_t n_ex = c->n_ex;
  CML_REQUIRE(x->state_arc_off[0] == 0 && x->state_arc_off[Q] == n_arcs, CML_ERR_ARG,
              "cml_build_trellises: state_arc_off must run from 0 to n_arcs");
  for (uint32_t s = 0; s < Q; ++s)
    CML_REQUIRE(x->state_arc_off[s] <= x->state_arc_off[s + 1], CML_ERR_ARG, "cml_build_trellises: state_arc_off not monotone");
  for (uint64_t a = 0; a < n_arcs; ++a)
    CML_REQUIRE(x->arc_dest[a] < Q, CML_ERR_ARG, "cml_build_trellises: arc destination out of range");
  for (uint64_t e = 0; e < n_ex; ++e)
    CML_REQUIRE(c->in_off[e] <= c->in_off[e + 1] && c->out_off[e] <= c->out_off[e + 1], CML_ERR_ARG,
                "cml_build_trellises: corpus offsets not monotone");
  // ---- (in,out)-label index of the transducer: per state the arc-table ids grouped by label pair, groups in key order,
  // ids of a group in arc-table order
  std::vector<uint32_t> state_off(Q + 1, 0), range_begin, ids;
  std::vector<uint64_t> keys;
  {
    std::vector<std::pair<uint64_t, uint32_t>> tmp;
    ids.reserve(n_arcs);
    for (uint32_t s = 0; s < Q; ++s) {
      tmp.clear();
      for (uint32_t a = x->state_arc_off[s]; a < x->state_arc_off[s + 1]; ++a)
        tmp.emplace_back(((uint64_t)x->arc_in[a] << 32) | x->arc_out[a], a);
      std::stable_sort(tmp.begin(), tmp.end(), [](auto const& p, auto const& q) { return p.first < q.first; });
      for (size_t i = 0; i < tmp.size(); ++i) {
        if (i == 0 || tmp[i].first != tmp[i - 1].first) {
          keys.push_back(tmp[i].first);
          range_begin.push_back((uint32_t)ids.size());
        }
        ids.push_back(tmp[i].second);
      }
      state_off[s + 1] = (uint32_t)keys.size();
    }
    range_begin.push_back((uint32_t)ids.size());
  }
  DevArray<uint32_t> d_state_off, d_range_begin, d_ids, d_dest, d_in_sym, d_out_sym, d_todo;
  DevArray<uint64_t> d_keys, d_in_off, d_out_off;
  CML_CUDA(d_state_off.upload(state_off.data(), state_off.size(), st));
  CML_CUDA(d_keys.upload(keys.data(), keys.size(), st));
  CML_CUDA(d_range_begin.upload(range_begin.data(), range_begin.size(), st));
  CML_CUDA(d_ids.upload(ids.data(), ids.size(), st));
  CML_CUDA(d_dest.upload(x->arc_dest, n_arcs, st));
  const uint64_t n_in = n_ex ? c->in_off[n_ex] : 0, n_out = n_ex ? c->out_off[n_ex] : 0;
  static const uint64_t zero1[1] = {0};
  CML_CUDA(d_in_off.upload(n_ex ? c->in_off : zero1, n_ex + 1, st));
  CML_CUDA(d_out_off.upload(n_ex ? c->out_off : zero1, n_ex + 1, st));
  CML_CUDA(d_in_sym.upload(c->in_sym, n_in, st));
  CML_CUDA(d_out_sym.upload(c->out_sym, n_out, st));
  DevArray<uint8_t> d_status;
  DevArray<uint32_t> d_nst, d_narc, d_fin, d_peak;
  DevArray<unsigned long long> d_next, d_pre;
  CML_CUDA(d_status.alloc(n_ex + 1));
  CML_CUDA(d_nst.alloc(n_ex + 1));
  CML_CUDA(d_narc.alloc(n_ex + 1));
  CML_CUDA(d_fin.alloc(n_ex + 1));
  CML_CUDA(d_peak.alloc(3));
  CML_CUDA(d_next.alloc(1));
  CML_CUDA(d_pre.alloc(1));
  CML_CUDA(cudaMemsetAsync(d_peak.p, 0, 3 * sizeof(uint32_t), st));
  CML_CUDA(cudaMemsetAsync(d_pre.p, 0, sizeof(unsigned long long), st));
  CML_CUDA(cudaMemsetAsync(d_status.p, B_OVERFLOW, n_ex + 1, st));

  size_t budget = (size_t)8 << 30;  // scratch bytes of one launch
  if (const char* e = getenv("CML_BUILD_SCRATCH_MB")) budget = (size_t)std::strtoull(e, nullptr, 10) << 20;
  const uint32_t max_workers = (uint32_t)ctx->sm_count * 2048u;
  auto per_worker = [](uint64_t C, uint64_t K, uint64_t M) {
    return M * sizeof(BSlot) + C + C * sizeof(BFrame) + K * sizeof(BKept) + C * 4 + (C + 1) * 4;
  };
  // one launch over `todo` with capacities (C, K); fill = pass 2
  auto launch = [&](std::vector<uint32_t> const& todo, uint64_t C, uint64_t K, int fill, const uint64_t* row_base, const uint64_t* arc_base,
                    uint32_t* o_off, uint32_t* o_dst, uint32_t* o_id) -> int {
    uint64_t M = 64;
    while (M < 2 * C) M <<= 1;
    uint64_t W = std::min<uint64_t>(std::min<uint64_t>(todo.size(), max_workers), std::max<uint64_t>(1, budget / per_worker(C, K, M)));
    W = (W + 127) / 128 * 128;
    ScopedDev<BSlot> map;
    ScopedDev<uint8_t> dead;
    ScopedDev<BFrame> stack;
    ScopedDev<BKept> kept;
    ScopedDev<uint32_t> renum, cnt;
    CML_CUDA(map.alloc(W * M));
    CML_CUDA(dead.alloc(W * C));
    CML_CUDA(stack.alloc(W * C));
    CML_CUDA(kept.alloc(W * K));
    CML_CUDA(renum.alloc(W * C));
    CML_CUDA(cnt.alloc(W * (C + 1)));
    CML_CUDA(cudaMemsetAsync(map.p, 0, W * M * sizeof(BSlot), st));
    CML_CUDA(d_todo.upload(todo.data(), todo.size(), st));
    CML_CUDA(cudaMemsetAsync(d_next.p, 0, sizeof(unsigned long long), st));
    BArgs A{};
    A.io = BIo{d_state_off.p, d_keys.p, d_range_begin.p, d_ids.p, d_dest.p, x->final_state};
    A.c = BCorpus{d_in_off.p, d_in_sym.p, d_out_off.p, d_out_sym.p};
    A.todo = d_todo.p;
    A.n_todo = (uint32_t)todo.size();
    A.C = (uint32_t)C;
    A.K = (uint32_t)K;
    A.mask = (uint32_t)(M - 1);
    A.map = map.p;
    A.dead = dead.p;
    A.stack = stack.p;
    A.kept = kept.p;
    A.renum = renum.p;
    A.cnt = cnt.p;
    A.next = d_next.p;
    A.status = d_status.p;
    A.n_states = d_nst.p;
    A.n_arcs = d_narc.p;
    A.fin = d_fin.p;
    A.peak = d_peak.p;
    A.pre_arcs = d_pre.p;
    A.fill = fill;
    A.row_base = row_base;
    A.arc_base = arc_base;
    A.out_off = o_off;
    A.out_dst = o_dst;
    A.out_id = o_id;
    k_build_trellis<<<(unsigned)(W / 128), 128, 0, st>>>(A);
    ++ctx->launches;
    CML_CUDA(cudaGetLastError());
    CML_CUDA(cudaStreamSynchronize(st));  // (the scratch is released on return)
    return CML_OK;
  };

  // ---- pass 1: sizes.  First capacity guess from the longest example; overflowing examples go to the next round.
  std::vector<uint8_t> status(n_ex + 1, B_OVERFLOW);
  std::vector<uint32_t> todo(n_ex);
  std::iota(todo.begin(), todo.end(), 0u);
  uint64_t max_len = 0;
  for (uint64_t e = 0; e < n_ex; ++e)
    max_len = std::max<uint64_t>(max_len, (c->in_off[e + 1] - c->in_off[e]) + (c->out_off[e + 1] - c->out_off[e]));
  uint64_t C = std::max<uint64_t>(64, (max_len + 2) * std::min<uint32_t>(Q, 8u));
  if (const char* e = getenv("CML_BUILD_FIRST_STATES")) C = std::max<uint64_t>(2, std::strtoull(e, nullptr, 10));
  uint64_t K = 8 * C;
  uint32_t rounds = 0;
  while (!todo.empty()) {
    CML_REQUIRE(per_worker(C, K, 4 * C) <= budget && C < (1ull << 30), CML_ERR_ARG,
                "cml_build_trellises: an example's lattice does not fit the scratch budget (CML_BUILD_SCRATCH_MB)");
    const int rc = launch(todo, C, K, 0, nullptr, nullptr, nullptr, nullptr, nullptr);
    if (rc) return rc;
    ++rounds;
    CML_CUDA(cudaMemcpy(status.data(), d_status.p, n_ex, cudaMemcpyDeviceToHost));
    std::vector<uint32_t> again;
    for (uint32_t e : todo) {
      CML_REQUIRE(status[e] != B_TOOLONG, CML_ERR_ARG, "cml_build_trellises: a string is longer than 65,534 symbols");
      if (status[e] == B_OVERFLOW) again.push_back(e);
    }
    todo.swap(again);
    // the overflowing walks stopped early: their peaks are lower bounds, so grow geometrically
    C *= 4;
    K *= 4;
  }
  std::unique_ptr<BuiltOwner> own(new BuiltOwner());
  std::vector<uint32_t> nst(n_ex), narc(n_ex), fin(n_ex);
  uint32_t peak[3] = {0, 0, 0};
  unsigned long long pre = 0;
  if (n_ex) {
    CML_CUDA(cudaMemcpy(nst.data(), d_nst.p, n_ex * 4, cudaMemcpyDeviceToHost));
    CML_CUDA(cudaMemcpy(narc.data(), d_narc.p, n_ex * 4, cudaMemcpyDeviceToHost));
    CML_CUDA(cudaMemcpy(fin.data(), d_fin.p, n_ex * 4, cudaMemcpyDeviceToHost));
  }
  CML_CUDA(cudaMemcpy(peak, d_peak.p, sizeof(peak), cudaMemcpyDeviceToHost));
  CML_CUDA(cudaMemcpy(&pre, d_pre.p, sizeof(pre), cudaMemcpyDeviceToHost));
  std::vector<uint64_t> row_base(n_ex + 1, 0), arc_base(n_ex + 1, 0);
  uint64_t rows = 0, arcs = 0;
  for (uint64_t e = 0; e < n_ex; ++e) {
    row_base[e] = rows;
    arc_base[e] = arcs;
    if (status[e] == B_OK) {
      own->kept_example.push_back((uint32_t)e);
      own->ex_states.push_back(nst[e]);
      own->ex_fin.push_back(fin[e]);
      own->ex_weight.push_back(c->weight ? c->weight[e] : 1.0);
      rows += (uint64_t)nst[e] + 1;
      arcs += narc[e];
    } else
      own->dropped.push_back((uint32_t)e);
  }
  // ---- pass 2: the kept examples again, rows and arcs written at their final places
  own->arc_off.resize(rows);
  own->arc_dst.resize(arcs);
  own->arc_id.resize(arcs);
  if (!own->kept_example.empty()) {
    DevArray<uint64_t> d_row_base, d_arc_base;
    DevArray<uint32_t> d_off, d_dst, d_id;
    CML_CUDA(d_row_base.upload(row_base.data(), n_ex + 1, st));
    CML_CUDA(d_arc_base.upload(arc_base.data(), n_ex + 1, st));
    CML_CUDA(d_off.alloc(rows));
    CML_CUDA(d_dst.alloc(std::max<uint64_t>(1, arcs)));
    CML_CUDA(d_id.alloc(std::max<uint64_t>(1, arcs)));
    const int rc = launch(own->kept_example, (uint64_t)peak[0] + 1, std::max<uint64_t>(1, peak[1]), 1, d_row_base.p, d_arc_base.p, d_off.p,
                          d_dst.p, d_id.p);
    if (rc) return rc;
    ++rounds;
    CML_CUDA(cudaMemcpy(own->arc_off.data(), d_off.p, rows * 4, cudaMemcpyDeviceToHost));
    if (arcs) {
      CML_CUDA(cudaMemcpy(own->arc_dst.data(), d_dst.p, arcs * 4, cudaMemcpyDeviceToHost));
      CML_CUDA(cudaMemcpy(own->arc_id.data(), d_id.p, arcs * 4, cudaMemcpyDeviceToHost));
    }
  }
  cml_built_trellises& P = own->pub;
  std::memset(&P, 0, sizeof(P));
  P.batch.n_ex = own->kept_example.size();
  P.batch.ex_states = own->ex_states.data();
  P.batch.ex_fin = own->ex_fin.data();
  P.batch.ex_weight = own->ex_weight.data();
  P.batch.arc_off = own->arc_off.data();
  P.batch.arc_dst = own->arc_dst.data();
  P.batch.arc_id = own->arc_id.data();
  P.kept_example = own->kept_example.data();
  P.n_dropped = own->dropped.size();
  P.dropped = own->dropped.data();
  P.pre_arcs = pre;
  P.launches = rounds;
  P.peak_states = peak[0];
  P.peak_kept_arcs = peak[1];
  P.peak_depth = peak[2];
  P.seconds = std::chrono::duration<double>(std::chrono::steady_clock::now() - t_start).count();
  P.owner = own.get();
  *out = &own.release()->pub;
  return CML_OK;
}

extern "C" int cml_build_free_trellises(cml_ctx* ctx, const cml_wfst_view* x, const cml_string_batch* sb, int given_tape,
                                        cml_built_trellises** out) {
  if (!ctx) return CML_ERR_ARG;
  CML_REQUIRE(x && sb && out, CML_ERR_ARG, "cml_build_free_trellises: null argument");
  *out = nullptr;
  CML_REQUIRE(given_tape == 0 || given_tape == 1, CML_ERR_ARG, "cml_build_free_trellises: the given tape must be 0 (input) or 1 (output)");
  CML_REQUIRE(x->n_states >= 1 && x->state_arc_off && (x->n_arcs == 0 || (x->arc_in && x->arc_out && x->arc_dest)), CML_ERR_ARG,
              "cml_build_free_trellises: incomplete transducer view");
  CML_REQUIRE(x->final_state < x->n_states, CML_ERR_ARG, "cml_build_free_trellises: final state out of range");
  CML_REQUIRE(x->n_arcs < 0xFFFFFFFFull, CML_ERR_ARG, "cml_build_free_trellises: too many arcs");
  const auto t_start = std::chrono::steady_clock::now();
  const uint32_t Q = x->n_states;
  const uint64_t n_arcs = x->n_arcs, n = sb->n;
  CML_REQUIRE(x->state_arc_off[0] == 0 && x->state_arc_off[Q] == n_arcs, CML_ERR_ARG,
              "cml_build_free_trellises: state_arc_off must run from 0 to n_arcs");
  for (uint32_t q = 0; q < Q; ++q)
    CML_REQUIRE(x->state_arc_off[q] <= x->state_arc_off[q + 1], CML_ERR_ARG, "cml_build_free_trellises: state_arc_off not monotone");
  for (uint64_t a = 0; a < n_arcs; ++a)
    CML_REQUIRE(x->arc_dest[a] < Q, CML_ERR_ARG, "cml_build_free_trellises: arc destination out of range");
  CML_REQUIRE(n < 0xFFFFFFFFull, CML_ERR_ARG, "cml_build_free_trellises: too many strings");
  CML_REQUIRE(n == 0 || (sb->off && sb->off[0] == 0 && (sb->off[n] == 0 || sb->sym)), CML_ERR_ARG,
              "cml_build_free_trellises: incomplete string batch (off[0] must be 0)");
  for (uint64_t e = 0; e < n; ++e) {
    CML_REQUIRE(sb->off[e] <= sb->off[e + 1], CML_ERR_ARG, "cml_build_free_trellises: string offsets not monotone");
    CML_REQUIRE((sb->off[e + 1] - sb->off[e] + 1) * Q < 0xFFFFFFFFull, CML_ERR_ARG,
                "cml_build_free_trellises: a string's lattice would have more than 2^32 states");
    // (|s| + 1) * n_arcs bounds the lattice's arcs, which the kernel counts in 32 bits (and arc_off holds)
    CML_REQUIRE((sb->off[e + 1] - sb->off[e] + 1) * n_arcs < 0xFFFFFFFFull, CML_ERR_ARG,
                "cml_build_free_trellises: a string's lattice could have more than 2^32 arcs");
  }
  const uint32_t* glab = given_tape == 0 ? x->arc_in : x->arc_out;
  // ---- eps-levels: longest-path depth in the subgraph of the arcs with *e* on the given tape (Kahn's order)
  std::vector<uint32_t> level(Q, 0), indeg(Q, 0), topo;
  for (uint64_t a = 0; a < n_arcs; ++a)
    if (glab[a] == 0) ++indeg[x->arc_dest[a]];
  topo.reserve(Q);
  for (uint32_t q = 0; q < Q; ++q)
    if (!indeg[q]) topo.push_back(q);
  for (size_t i = 0; i < topo.size(); ++i) {
    const uint32_t q = topo[i];
    for (uint32_t a = x->state_arc_off[q]; a < x->state_arc_off[q + 1]; ++a) {
      if (glab[a] != 0) continue;
      const uint32_t d = x->arc_dest[a];
      level[d] = std::max(level[d], level[q] + 1);
      if (--indeg[d] == 0) topo.push_back(d);
    }
  }
  CML_REQUIRE(topo.size() == Q, CML_ERR_CYCLE,
              std::string("cml_build_free_trellises: the arcs with *e* on the given ") + (given_tape ? "output" : "input") +
                  " tape form a cycle, so a string would have unboundedly many derivations (given-*e* cycles are not decoded)");
  std::vector<uint32_t> order(Q);
  std::iota(order.begin(), order.end(), 0u);
  std::stable_sort(order.begin(), order.end(), [&](uint32_t a, uint32_t b) { return level[a] < level[b]; });
  const uint32_t L = level[order.back()] + 1;
  std::vector<uint32_t> lvl_off(L + 1, 0);
  for (uint32_t q = 0; q < Q; ++q) ++lvl_off[level[q] + 1];
  for (uint32_t l = 0; l < L; ++l) lvl_off[l + 1] += lvl_off[l];
  // ---- given-symbol index: per state the arc-table ids grouped by given-tape symbol, groups ascending, ids of a group
  // in arc-table order
  std::vector<uint32_t> key_off(Q + 1, 0), keys, grp, ids;
  {
    std::vector<std::pair<uint32_t, uint32_t>> tmp;
    ids.reserve(n_arcs);
    for (uint32_t q = 0; q < Q; ++q) {
      tmp.clear();
      for (uint32_t a = x->state_arc_off[q]; a < x->state_arc_off[q + 1]; ++a) tmp.emplace_back(glab[a], a);
      std::stable_sort(tmp.begin(), tmp.end(), [](auto const& p, auto const& r) { return p.first < r.first; });
      for (size_t i = 0; i < tmp.size(); ++i) {
        if (i == 0 || tmp[i].first != tmp[i - 1].first) {
          keys.push_back(tmp[i].first);
          grp.push_back((uint32_t)ids.size());
        }
        ids.push_back(tmp[i].second);
      }
      key_off[q + 1] = (uint32_t)keys.size();
    }
    grp.push_back((uint32_t)ids.size());
  }
  // ---- chunks of consecutive strings whose cells (6 B each) fit the budget
  const uint64_t budget = (uint64_t)ctx->opt_free_build_scratch_mb << 20;
  std::vector<uint64_t> cell_base(n + 1, 0), chunk_begin(1, 0);
  uint64_t cells = 0, max_cells = 0;
  for (uint64_t e = 0; e < n; ++e) {
    const uint64_t c = (sb->off[e + 1] - sb->off[e] + 1) * Q;
    if (cells && (cells + c) * 6 > budget) {
      chunk_begin.push_back(e);
      max_cells = std::max(max_cells, cells);
      cells = 0;
    }
    cell_base[e] = cells;
    cells += c;
  }
  max_cells = std::max(max_cells, cells);
  chunk_begin.push_back(n);
  const uint64_t n_chunks = chunk_begin.size() - 1;

  CML_CUDA(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  DevArray<uint32_t> d_key_off, d_keys, d_grp, d_ids, d_dest, d_order, d_lvl_off, d_sym, d_nst, d_narc;
  DevArray<uint64_t> d_soff, d_cell_base, d_row_base, d_arc_base;
  DevArray<uint8_t> d_fw, d_kept;
  DevArray<uint32_t> d_id, d_off, d_dst, d_aid;
  CML_CUDA(d_key_off.upload(key_off.data(), key_off.size(), st));
  CML_CUDA(d_keys.upload(keys.data(), keys.size(), st));
  CML_CUDA(d_grp.upload(grp.data(), grp.size(), st));
  CML_CUDA(d_ids.upload(ids.data(), ids.size(), st));
  CML_CUDA(d_dest.upload(x->arc_dest, n_arcs, st));
  CML_CUDA(d_order.upload(order.data(), Q, st));
  CML_CUDA(d_lvl_off.upload(lvl_off.data(), lvl_off.size(), st));
  static const uint64_t zero1[1] = {0};
  CML_CUDA(d_soff.upload(n ? sb->off : zero1, n + 1, st));
  CML_CUDA(d_sym.upload(sb->sym, n ? sb->off[n] : 0, st));
  CML_CUDA(d_cell_base.upload(cell_base.data(), n + 1, st));
  CML_CUDA(d_nst.alloc(n + 1));
  CML_CUDA(d_narc.alloc(n + 1));
  CML_CUDA(d_row_base.alloc(n + 1));
  CML_CUDA(d_arc_base.alloc(n + 1));
  CML_CUDA(d_fw.alloc(std::max<uint64_t>(1, max_cells)));
  CML_CUDA(d_kept.alloc(std::max<uint64_t>(1, max_cells)));
  CML_CUDA(d_id.alloc(std::max<uint64_t>(1, max_cells)));
  EventPair ev;
  CML_CUDA(ev.create());

  std::unique_ptr<BuiltOwner> own(new BuiltOwner());
  std::vector<uint32_t> nst(n + 1), narc(n + 1);
  std::vector<uint64_t> row_base(n + 1, 0), arc_base(n + 1, 0);
  uint32_t launches = 0, peak_states = 0, peak_arcs = 0;
  double kernel_ms = 0;
  FArgs A{};
  A.key_off = d_key_off.p;
  A.keys = d_keys.p;
  A.grp = d_grp.p;
  A.ids = d_ids.p;
  A.dest = d_dest.p;
  A.order = d_order.p;
  A.lvl_off = d_lvl_off.p;
  A.Q = Q;
  A.L = L;
  A.final_state = x->final_state;
  A.s_off = d_soff.p;
  A.sym = d_sym.p;
  A.cell_base = d_cell_base.p;
  A.fw = d_fw.p;
  A.kept = d_kept.p;
  A.id = d_id.p;
  A.n_st = d_nst.p;
  A.n_arc = d_narc.p;
  A.row_base = d_row_base.p;
  A.arc_base = d_arc_base.p;
  const unsigned max_blocks = (unsigned)ctx->sm_count * 16u;
  for (uint64_t c = 0; c < n_chunks; ++c) {
    const uint64_t e0 = chunk_begin[c], e1 = chunk_begin[c + 1];
    if (e0 == e1) continue;
    const uint64_t chunk_cells = (e1 < n ? cell_base[e1 - 1] + (sb->off[e1] - sb->off[e1 - 1] + 1) * Q : cells);
    CML_CUDA(cudaMemsetAsync(d_fw.p, 0, chunk_cells, st));
    A.e0 = e0;
    A.n_list = (uint32_t)(e1 - e0);
    const unsigned grid = std::max(1u, std::min(cdiv(e1 - e0, kFreeWarps), max_blocks));
    float ms = 0;
    // pass 0: reachability, ids, sizes
    A.fill = 0;
    CML_CUDA(cudaEventRecord(ev.a, st));
    k_build_free<<<grid, kFreeWarps * 32, 0, st>>>(A);
    CML_CUDA(cudaGetLastError());
    CML_CUDA(cudaEventRecord(ev.b, st));
    ++launches;
    ++ctx->launches;
    CML_CUDA(cudaMemcpyAsync(nst.data() + e0, d_nst.p + e0, (e1 - e0) * 4, cudaMemcpyDeviceToHost, st));
    CML_CUDA(cudaMemcpyAsync(narc.data() + e0, d_narc.p + e0, (e1 - e0) * 4, cudaMemcpyDeviceToHost, st));
    CML_CUDA(cudaStreamSynchronize(st));
    CML_CUDA(cudaEventElapsedTime(&ms, ev.a, ev.b));
    kernel_ms += ms;
    // exclusive scan of the kept lattices' sizes: their places in the chunk's output
    uint64_t rows = 0, arcs = 0;
    for (uint64_t e = e0; e < e1; ++e) {
      row_base[e] = rows;
      arc_base[e] = arcs;
      if (nst[e]) {
        rows += (uint64_t)nst[e] + 1;
        arcs += narc[e];
        peak_states = std::max(peak_states, nst[e]);
        peak_arcs = std::max(peak_arcs, narc[e]);
      }
    }
    if (!rows) {
      for (uint64_t e = e0; e < e1; ++e) own->dropped.push_back((uint32_t)e);
      continue;
    }
    // pass 1: rows and arcs at their places (the cells of pass 0 are still in the scratch)
    CML_CUDA(cudaMemcpyAsync(d_row_base.p + e0, row_base.data() + e0, (e1 - e0) * 8, cudaMemcpyHostToDevice, st));
    CML_CUDA(cudaMemcpyAsync(d_arc_base.p + e0, arc_base.data() + e0, (e1 - e0) * 8, cudaMemcpyHostToDevice, st));
    if (d_off.n < rows) CML_CUDA(d_off.alloc(rows));
    if (d_dst.n < std::max<uint64_t>(1, arcs)) {
      CML_CUDA(d_dst.alloc(std::max<uint64_t>(1, arcs)));
      CML_CUDA(d_aid.alloc(std::max<uint64_t>(1, arcs)));
    }
    A.fill = 1;
    A.out_off = d_off.p;
    A.out_dst = d_dst.p;
    A.out_id = d_aid.p;
    CML_CUDA(cudaEventRecord(ev.a, st));
    k_build_free<<<grid, kFreeWarps * 32, 0, st>>>(A);
    CML_CUDA(cudaGetLastError());
    CML_CUDA(cudaEventRecord(ev.b, st));
    ++launches;
    ++ctx->launches;
    const size_t r0 = own->arc_off.size(), a0 = own->arc_dst.size();
    own->arc_off.resize(r0 + rows);
    own->arc_dst.resize(a0 + arcs);
    own->arc_id.resize(a0 + arcs);
    CML_CUDA(cudaMemcpyAsync(own->arc_off.data() + r0, d_off.p, rows * 4, cudaMemcpyDeviceToHost, st));
    if (arcs) {
      CML_CUDA(cudaMemcpyAsync(own->arc_dst.data() + a0, d_dst.p, arcs * 4, cudaMemcpyDeviceToHost, st));
      CML_CUDA(cudaMemcpyAsync(own->arc_id.data() + a0, d_aid.p, arcs * 4, cudaMemcpyDeviceToHost, st));
    }
    CML_CUDA(cudaStreamSynchronize(st));
    CML_CUDA(cudaEventElapsedTime(&ms, ev.a, ev.b));
    kernel_ms += ms;
    for (uint64_t e = e0; e < e1; ++e) {
      if (!nst[e]) {
        own->dropped.push_back((uint32_t)e);
        continue;
      }
      own->kept_example.push_back((uint32_t)e);
      own->ex_states.push_back(nst[e]);
      own->ex_fin.push_back(nst[e] - 1);
      own->ex_weight.push_back(1.0);
    }
  }
  cml_built_trellises& P = own->pub;
  std::memset(&P, 0, sizeof(P));
  P.batch.n_ex = own->kept_example.size();
  P.batch.ex_states = own->ex_states.data();
  P.batch.ex_fin = own->ex_fin.data();
  P.batch.ex_weight = own->ex_weight.data();
  P.batch.arc_off = own->arc_off.data();
  P.batch.arc_dst = own->arc_dst.data();
  P.batch.arc_id = own->arc_id.data();
  P.kept_example = own->kept_example.data();
  P.n_dropped = own->dropped.size();
  P.dropped = own->dropped.data();
  P.launches = launches;
  P.peak_states = peak_states;
  P.peak_kept_arcs = peak_arcs;
  P.chunks = n_chunks;
  P.kernel_ms = kernel_ms;
  P.seconds = std::chrono::duration<double>(std::chrono::steady_clock::now() - t_start).count();
  P.owner = own.get();
  *out = &own.release()->pub;
  return CML_OK;
}

extern "C" void cml_free_built_trellises(cml_built_trellises* b) {
  if (b && b->owner) delete static_cast<BuiltOwner*>(b->owner);
}
