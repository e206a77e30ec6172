// cml_forest.cu -- forest-em's inside-outside E-step and NormalizeGroups M-step on the GPU (sm_100a).
//
// Reference path (SURVEY.md section 8 rows a19-a23): FForest::inside_rec / compute_norm_outside /
// visit_inside_norm_outside (forest-em/forest.hpp:326-491,636-697), FForests::estimate / maximize
// (forest-em/forest-em.hpp:511-572,626-655), NormalizeGroups (graehl/shared/normalize.hpp:123-164).
//
// Layout in HBM.  Three families (cml_forests_set_layout): level-synchronous tiles -- a CTA owns a run of forests, nodes
// height-major across them, all values in shared memory (k_forest_level, the throughput path, described at the kernel);
// per-forest height-levelised CSRs (k_forest_warp / k_forest_cta, described here); thread-per-forest streams
// (k_forest_thread).  A forest arrives as the reference's pre-order node array.  Here back references are
// resolved (a shared node is ONE node with several parents), the real nodes are sorted by height
// (leaves = 0; a parent is strictly higher than its children), and the hyperedges are stored as two
// CSRs over that order: children (inside pass, ascending height) and parents (outside pass, descending
// height).  Per node: label u32 (rule id, 0 = OR; bit 31 marks a "hot" rule), child_off u32, par_off u32;
// per child/parent link: u32 node index (parent links carry the parent's OR flag in bit 31).
//
// Arithmetic.  inside[] is a natural log in fp32/fp64 with the reference's log-add (cutoff 16/36 nats,
// sequential over the OR children in the reference's order).  The outside pass does not keep
// norm_outside = outside/inside[root] (range of a log) but the posterior gamma[n] = inside[n]*norm_outside[n]
// in [0, ~1], in linear space: AND parent -> child adds gamma[p]; OR parent -> child adds
// gamma[p]*exp(inside[c]-inside[p]).  It is a pull over the parent CSR: no atomics, deterministic.
// counts[rule] += gamma[n] for AND nodes: fp64 RED into an L2-resident table; rules that occur very
// often are accumulated in 64 replicated slots first (see k_forest_fold) to keep one address from
// serialising the whole GPU.
#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstring>
#include <memory>
#include <thread>

#include "cml_common.cuh"

namespace {

const uint32_t kHotBit = 0x80000000u;
const int kHotCopies = 64;
const int kWarpsPerCta = 4;
const int kNWarpCls = 6;
const uint32_t kWarpCaps[kNWarpCls] = {128, 256, 512, 1024, 2048, 4096};  // nodes per forest, shared memory classes
const int kCtaThreads = 256;

struct __align__(16) ForestDesc {
  uint64_t node_base;  // first entry in label / child_off / par_off (n_nodes + 1 entries each, own sentinel)
  uint64_t child_base, par_base;  // first link of this forest in child / par
  uint64_t lvl_base;   // first entry (n_levels + 1) in lvl_off
  uint32_t n_nodes, n_levels;
  uint32_t index;      // forest number within its batch (for ln_inside)
  uint32_t pad;
};

template <typename Real>
struct FNum;
template <>
struct FNum<float> {
  static __device__ __forceinline__ float ninf() { return -CUDART_INF_F; }
  static __device__ __forceinline__ float cut() { return 16.f; }
  static __device__ __forceinline__ float ex(float x) { return __expf(x); }
  static __device__ __forceinline__ float exa(float x) { return expf(x); }
  static __device__ __forceinline__ float l1p(float x) { return log1pf(x); }
};
template <>
struct FNum<double> {
  static __device__ __forceinline__ double ninf() { return -CUDART_INF; }
  static __device__ __forceinline__ double cut() { return 36.; }
  static __device__ __forceinline__ double ex(double x) { return exp(x); }
  static __device__ __forceinline__ double exa(double x) { return exp(x); }
  static __device__ __forceinline__ double l1p(double x) { return log1p(x); }
};
// logweight operator+ (graehl/shared/weight.h:765-801)
template <typename Real>
__device__ __forceinline__ Real ln_add(Real a, Real b) {
  if (!(a > FNum<Real>::ninf())) return b;
  if (!(b > FNum<Real>::ninf())) return a;
  const Real d = a - b;
  if (d > FNum<Real>::cut()) return a;
  if (d < -FNum<Real>::cut()) return b;
  return d < 0 ? b + FNum<Real>::l1p(FNum<Real>::exa(d)) : a + FNum<Real>::l1p(FNum<Real>::exa(-d));
}

struct ForestArgs {
  const ForestDesc* desc;
  const uint32_t* list;  // forests of this launch (indices into desc)
  uint32_t n_list;
  const uint32_t* label;
  const uint32_t* child_off;
  const uint32_t* par_off;
  const uint32_t* child;
  const uint32_t* par;
  const uint32_t* lvl_off;
  const void* lnw;          // Real[rulespace]
  const uint32_t* hot_index;  // [rulespace] replica row of hot rules
  double* counts;           // [rulespace]
  double* hot;              // [kHotCopies][n_hot]
  uint32_t n_hot;
  double* ln_inside;        // per forest of the batch
  void* scratch;            // CTA class: Real[2 * scratch_stride] per block
  uint64_t scratch_stride;
  uint32_t cap;             // warp classes: node capacity per warp
};

template <int NT>
__device__ __forceinline__ void fsync() {
  if (NT == 32)
    __syncwarp();
  else
    __syncthreads();
}

// One forest by one group of NT threads.  in_/ga: NT-shared arrays of n_nodes values (shared or global).
template <typename Real, int NT>
__device__ void forest_inside_outside(const ForestArgs& A, const ForestDesc& d, Real* __restrict__ in_, Real* __restrict__ ga,
                                      int lane, uint32_t replica) {
  const uint32_t* __restrict__ label = A.label + d.node_base;
  const uint32_t* __restrict__ coff = A.child_off + d.node_base;
  const uint32_t* __restrict__ poff = A.par_off + d.node_base;
  const uint32_t* __restrict__ child = A.child + d.child_base;
  const uint32_t* __restrict__ par = A.par + d.par_base;
  const uint32_t* __restrict__ lvl = A.lvl_off + d.lvl_base;
  const Real* __restrict__ lnw = (const Real*)A.lnw;
  const uint32_t nl = d.n_levels;
  const Real NI = FNum<Real>::ninf();
  // ---- inside: ascending height (forest.hpp:636-697) ------------------------------------------------
  for (uint32_t L = 0; L < nl; ++L) {
    const uint32_t i1 = __ldg(&lvl[L + 1]);
    for (uint32_t i = __ldg(&lvl[L]) + lane; i < i1; i += NT) {
      const uint32_t lab = __ldg(&label[i]) & ~kHotBit;
      uint32_t c = __ldg(&coff[i]);
      const uint32_t c1 = __ldg(&coff[i + 1]);
      Real v;
      if (lab) {  // AND: rule weight times the children
        v = __ldg(&lnw[lab]);
        for (; c < c1; ++c) v += in_[__ldg(&child[c])];
      } else {    // OR: first child, then fold the rest in order
        v = in_[__ldg(&child[c])];
        for (++c; c < c1; ++c) v = ln_add<Real>(v, in_[__ldg(&child[c])]);
      }
      in_[i] = v;
    }
    fsync<NT>();
  }
  const uint32_t root = d.n_nodes - 1;  // the only node of the top level
  const Real in_root = in_[root];
  if (lane == 0) A.ln_inside[d.index] = (double)in_root;
  if (!(in_root > NI)) return;  // zero-probability forest: no counts (forest.hpp:447-451)
  // ---- outside as posteriors, descending height, pull over parents (forest.hpp:439-491) -------------
  for (uint32_t L = nl; L-- > 0;) {
    const uint32_t i1 = __ldg(&lvl[L + 1]);
    for (uint32_t i = __ldg(&lvl[L]) + lane; i < i1; i += NT) {
      Real g = i == root ? Real(1) : Real(0);
      const Real in_i = in_[i];
      uint32_t k = __ldg(&poff[i]);
      const uint32_t k1 = __ldg(&poff[i + 1]);
      for (; k < k1; ++k) {
        const uint32_t e = __ldg(&par[k]);
        const uint32_t p = e & ~kHotBit;
        const Real gp = ga[p];
        if (e & kHotBit) {  // OR parent: share of this alternative
          if (in_i > NI && gp > 0) g += gp * FNum<Real>::ex(in_i - in_[p]);
        } else
          g += gp;          // AND parent: every child is used whenever the parent is
      }
      ga[i] = g;
      const uint32_t lab = __ldg(&label[i]);
      if ((lab & ~kHotBit) && g > 0) {
        if (lab & kHotBit)
          atomicAdd(A.hot + (size_t)replica * A.n_hot + __ldg(&A.hot_index[lab & ~kHotBit]), (double)g);
        else
          atomicAdd(A.counts + lab, (double)g);
      }
    }
    fsync<NT>();
  }
}

template <typename Real>
__global__ void __launch_bounds__(kWarpsPerCta * 32) k_forest_warp(ForestArgs A) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  Real* in_ = (Real*)smem_raw + (size_t)warp * 2 * A.cap;
  Real* ga = in_ + A.cap;
  const uint32_t gw = blockIdx.x * kWarpsPerCta + warp, nw = gridDim.x * kWarpsPerCta;
  for (uint32_t f = gw; f < A.n_list; f += nw) {
    const ForestDesc d = A.desc[A.list[f]];
    forest_inside_outside<Real, 32>(A, d, in_, ga, lane, gw & (kHotCopies - 1));
    __syncwarp();
  }
}

template <typename Real>
__global__ void __launch_bounds__(kCtaThreads) k_forest_cta(ForestArgs A) {
  Real* in_ = (Real*)A.scratch + (size_t)blockIdx.x * 2 * A.scratch_stride;
  Real* ga = in_ + A.scratch_stride;
  for (uint32_t f = blockIdx.x; f < A.n_list; f += gridDim.x) {
    const ForestDesc d = A.desc[A.list[f]];
    forest_inside_outside<Real, kCtaThreads>(A, d, in_, ga, threadIdx.x, blockIdx.x & (kHotCopies - 1));
    __syncthreads();
  }
}

// ---------------------------------------------------------------------------------------------------
// Thread-per-forest kernel (the throughput path for corpora of many small forests).
//
// 32 forests of similar size form a tile, one forest per lane of a warp; the two passes are flattened into
// streams of 32-bit words stored transposed ([row][lane]), so the warp's loads of its 32 sequential streams
// coalesce into one 128-byte line per row.  Nodes are numbered in DFS post-order (children before parents, the
// root last).  Per node a HEADER word (rule id, flags), then one word per link:
//   inside  stream: children;  a tree child (defined inside its parent) was completed just before and sits on
//                   top of the lane's VALUE STACK in shared memory: POP.  Only children reached through a back
//                   reference (shared sub-forests) are read from the global inside[] array.
//   outside stream: nodes in reverse post-order (= a pre-order walk), parents;  the tree parent is an ancestor on
//                   the current root-to-node path and sits in the lane's PATH STACK (gamma, inside) at depth-1:
//                   TREE.  Only the other parents of a shared node are read from the global gamma[] / inside[].
// (profiles/r1i_k_forest_thread_f32.txt: with every value read from global memory the kernel ran at 21 warps per SM
// with 31 cycles of long-scoreboard stall per issue -- one dependent, uncoalesced load per link.)
// Streams run through a per-warp cp.async ring in shared memory, two 8-row chunks ahead; rule weights one chunk ahead.  All lanes run the
// same trip count (rows of the largest forest of the tile; the rest is NOP padding) with no synchronisation.
// A forest whose text order is not a proper tree walk, or whose stacks would be deeper than the caps, simply
// carries no POP / TREE / PUSH flags and reads everything from global memory.
// ---------------------------------------------------------------------------------------------------
const uint32_t kOpNop = 0xffffffffu;
const uint32_t kHdr = 0x80000000u, kOpLast = 0x40000000u;
const uint32_t kHdrPush = 0x20000000u, kHdrDepthShift = 23, kHdrHot = 1u << 22, kHdrLabel = (1u << 22) - 1;
const uint32_t kHdrNparShift = 22;  // inside headers only: 7 bits (depth and hot are outside-stream fields)
const uint32_t kLinkPop = 0x20000000u, kLinkIdxIn = 0x1fffffffu;                       // inside links
const uint32_t kLinkOr = 0x20000000u, kLinkTree = 0x10000000u, kLinkIdxOut = 0x0fffffffu;  // outside links
const int kStackCap = 64, kDepthCap = 63, kTileU = 8, kTileStages = 3;  // rows per chunk; chunks in the cp.async ring (shared memory decides the resident warps)
const int kTileAhead = kTileStages + 1;  // chunks of NOP padding behind the streams (prefetch runs past the end)
struct __align__(16) TileDesc {
  uint64_t ops_in_base, ops_out_base, row_base;  // element offsets (already multiplied by 32) into t_ops_in / t_ops_out / rows
  uint32_t steps_in, steps_out;                  // multiples of kTileU
  uint32_t n_nodes[32];
  uint32_t forest[32];  // forest number within the batch, 0xffffffff = empty lane
  uint32_t rows_out[32];  // words of the lane's outside stream (nodes + links)
};
struct TileArgs {
  const TileDesc* tiles;
  uint32_t n_tiles;
  const uint32_t* ops_in;
  const uint32_t* ops_out;
  void* in_;              // Real [row][lane]
  void* ga;
  void* vout;             // Real [outside stream row][lane]: inside[node] at the row of the node's outside header
  const void* lnw;
  const uint32_t* hot_index;
  double* counts;
  double* hot;
  uint32_t n_hot;
  double* ln_inside;
  uint32_t stack_rows;    // shared-memory rows per lane: >= value-stack depth and >= 2 * (path depth + 1), even
};
template <typename Real>
__device__ __forceinline__ Real ln_add_fast(Real a, Real b);
template <>
__device__ __forceinline__ double ln_add_fast<double>(double a, double b) {
  return ln_add<double>(a, b);
}
template <>
__device__ __forceinline__ float ln_add_fast<float>(float a, float b) {  // same cutoff semantics, hardware exp/log
  if (!(a > -CUDART_INF_F)) return b;
  if (!(b > -CUDART_INF_F)) return a;
  const float hi = fmaxf(a, b), d = -fabsf(a - b);
  if (d < -16.f) return hi;
  return hi + __logf(1.f + __expf(d));
}
const int kTileWarps = 4;
__device__ __forceinline__ void f_cp_async4(uint32_t smem_dst, const void* gsrc) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;\n" ::"r"(smem_dst), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void f_cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::: "memory"); }
template <int BYTES>
__device__ __forceinline__ void f_cp_async_n(uint32_t smem_dst, const void* gsrc) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], %2;\n" ::"r"(smem_dst), "l"(gsrc), "n"(BYTES) : "memory");
}
template <int N>
__device__ __forceinline__ void f_cp_async_wait() {
  asm volatile("cp.async.wait_group %0;\n" ::"n"(N) : "memory");
}
template <typename Real>
__global__ void __launch_bounds__(kTileWarps * 32) k_forest_thread(TileArgs A) {
  extern __shared__ __align__(16) unsigned char smem_ft[];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const uint32_t t = blockIdx.x * kTileWarps + wib;
  if (t >= A.n_tiles) return;
  // per-lane columns: value stack (inside pass), then reused as the gamma / inside path stacks (outside pass)
  Real* stk = reinterpret_cast<Real*>(smem_ft) + (size_t)wib * A.stack_rows * 32 + lane;
  Real* gstk = stk;
  Real* istk = stk + (size_t)(A.stack_rows / 2) * 32;
  // the stream ring of this warp: kTileStages chunks of kTileU rows of 32 words, behind all the stacks
  uint32_t* ring_w = reinterpret_cast<uint32_t*>(reinterpret_cast<Real*>(smem_ft) + (size_t)kTileWarps * A.stack_rows * 32) +
                     (size_t)wib * kTileStages * kTileU * 32 + lane;
  const uint32_t sring = (uint32_t)__cvta_generic_to_shared(ring_w);
  // ... and the ring of inside values that travels with the outside stream (same rows)
  Real* vring = reinterpret_cast<Real*>(reinterpret_cast<uint32_t*>(reinterpret_cast<Real*>(smem_ft) +
                                                                      (size_t)kTileWarps * A.stack_rows * 32) +
                                         (size_t)kTileWarps * kTileStages * kTileU * 32) +
                (size_t)wib * kTileStages * kTileU * 32 + lane;
  const uint32_t svring = (uint32_t)__cvta_generic_to_shared(vring);
  const TileDesc* __restrict__ T = A.tiles + t;
  const uint32_t* __restrict__ oi = A.ops_in + T->ops_in_base + lane;
  const uint32_t* __restrict__ oo = A.ops_out + T->ops_out_base + lane;
  Real* __restrict__ in_ = (Real*)A.in_ + T->row_base + lane;
  Real* __restrict__ ga = (Real*)A.ga + T->row_base + lane;
  const Real* __restrict__ lnw = (const Real*)A.lnw;
  const Real NI = FNum<Real>::ninf();
  const uint32_t n = T->n_nodes[lane];
  const uint32_t fidx = T->forest[lane];
  const uint32_t replica = t & (kHotCopies - 1);
  auto hdr_weight = [&](uint32_t op) -> Real {  // rule weight of a header word (0 = OR / not a header: unused)
    const uint32_t lab = op & kHdrLabel;
    return ((op & kHdr) && op != kOpNop && lab) ? __ldg(&lnw[lab]) : NI;
  };
  // ---- inside
  uint32_t jn = 0, sp = 0, cum = 0;
  const uint32_t rows_out = T->rows_out[lane] & 0x7fffffffu;
  const bool use_vout = (T->rows_out[lane] >> 31) == 0;  // (a node with > 127 parents: read inside[] directly instead)
  Real* __restrict__ vo = (Real*)A.vout + T->ops_out_base + lane;
  Real v = NI;
  bool isand = false, push = false;
  {
    // The stream goes through a per-warp cp.async ring in shared memory, kTileStages - 1 chunks (of 8 rows) ahead:
    // register-staged prefetch stopped helping beyond one chunk because the loads share scoreboards and a rotating
    // move waits for the newest one (profiles/r1k, r1l).  A lane copies and later reads only its own words, so
    // cp.async.wait_group is all the synchronisation needed.  Rule weights of a chunk's headers are gathered one
    // chunk before its turn, into two register sets used alternately (the loop body handles two chunks).
    const uint32_t si = T->steps_in;  // multiple of 2 * kTileU
    auto issue = [&](uint32_t row) {  // queue chunk `row / kTileU` of the stream (rows past the end are NOP padding)
      const uint32_t st = (row / kTileU) % kTileStages;
#pragma unroll
      for (int k = 0; k < kTileU; ++k)
        f_cp_async4(sring + (uint32_t)((st * kTileU + k) * 32) * 4u, oi + (size_t)(row + k) * 32);
      f_cp_async_commit();
    };
    auto ops_of = [&](uint32_t row, uint32_t (&a)[kTileU]) {
      const uint32_t st = (row / kTileU) % kTileStages;
#pragma unroll
      for (int k = 0; k < kTileU; ++k) a[k] = ring_w[(st * kTileU + k) * 32];
    };
    auto weights = [&](const uint32_t (&a)[kTileU], Real (&w)[kTileU]) {
#pragma unroll
      for (int k = 0; k < kTileU; ++k) w[k] = hdr_weight(a[k]);
    };
    auto process = [&](const uint32_t (&a)[kTileU], const Real (&w)[kTileU]) {
#pragma unroll
      for (int k = 0; k < kTileU; ++k) {
        const uint32_t op = a[k];
        if (op == kOpNop) continue;
        if (op & kHdr) {
          isand = (op & kHdrLabel) != 0;
          push = (op & kHdrPush) != 0;
          cum += 1u + ((op >> kHdrNparShift) & 127u);  // words of this node in the outside stream: header + parents
          v = w[k];
        } else {
          Real x;
          if (op & kLinkPop)
            x = stk[(size_t)(--sp) * 32];
          else
            x = in_[(size_t)(op & kLinkIdxIn) * 32];
          v = isand ? v + x : ln_add_fast<Real>(v, x);
        }
        if (op & kOpLast) {
          in_[(size_t)jn * 32] = v;
          // the outside pass walks the nodes backwards: leave inside[node] where its stream will pass (the row of
          // the node's outside header), so that pass reads it through its prefetch ring and not with a dependent load
          if (use_vout) vo[(size_t)(rows_out - cum) * 32] = v;
          if (push) stk[(size_t)(sp++) * 32] = v;
          ++jn;
        }
      }
    };
    uint32_t oa[kTileU], ob[kTileU];
    Real wa[kTileU], wb[kTileU];
#pragma unroll
    for (int st = 0; st < kTileStages - 1; ++st) issue(st * kTileU);
    f_cp_async_wait<kTileStages - 2>();  // chunk 0 has landed
    ops_of(0, oa);
    weights(oa, wa);
    for (uint32_t s = 0; s < si; s += 2 * kTileU) {
      issue(s + (kTileStages - 1) * kTileU);
      f_cp_async_wait<kTileStages - 2>();  // chunk s/8 + 1 has landed
      ops_of(s + kTileU, ob);
      weights(ob, wb);
      process(oa, wa);
      issue(s + kTileStages * kTileU);
      f_cp_async_wait<kTileStages - 2>();  // chunk s/8 + 2
      ops_of(s + 2 * kTileU, oa);
      weights(oa, wa);
      process(ob, wb);
    }
    f_cp_async_wait<0>();
  }
  if (fidx == 0xffffffffu) return;
  const Real in_root = v;  // the root is the last node of the post-order
  A.ln_inside[fidx] = (double)in_root;
  if (!(in_root > NI)) return;  // zero-probability forests collect no counts (forest.hpp:447-451)
  // ---- outside as posteriors: reverse post-order
  {
    jn = n - 1;
    Real g = 0;
    uint32_t hdr = 0;
    Real in_i = NI;
    const uint32_t so = T->steps_out;  // multiple of kTileU
    uint32_t hidx = 0;
    auto issue = [&](uint32_t row) {  // the op stream and, row for row, the inside values the inside pass left
      const uint32_t st = (row / kTileU) % kTileStages;
#pragma unroll
      for (int k = 0; k < kTileU; ++k) {
        f_cp_async4(sring + (uint32_t)((st * kTileU + k) * 32) * 4u, oo + (size_t)(row + k) * 32);
        f_cp_async_n<sizeof(Real)>(svring + (uint32_t)((st * kTileU + k) * 32) * (uint32_t)sizeof(Real),
                                   vo + (size_t)(row + k) * 32);
      }
      f_cp_async_commit();
    };
    auto ops_of = [&](uint32_t row, uint32_t (&a)[kTileU], Real (&val)[kTileU]) {
      const uint32_t st = (row / kTileU) % kTileStages;
#pragma unroll
      for (int k = 0; k < kTileU; ++k) {
        a[k] = ring_w[(st * kTileU + k) * 32];
        val[k] = vring[(st * kTileU + k) * 32];
      }
    };
    auto process = [&](const uint32_t (&a)[kTileU], const Real (&val)[kTileU]) {
#pragma unroll
      for (int k = 0; k < kTileU; ++k) {
        const uint32_t op = a[k];
        if (op == kOpNop) continue;
        if (op & kHdr) {
          hdr = op;
          in_i = use_vout ? val[k] : in_[(size_t)jn * 32];
          g = (op & kOpLast) ? Real(1) : Real(0);  // a header that is also LAST has no parents: the root
          if (op & kHdrHot) hidx = __ldg(&A.hot_index[op & kHdrLabel]);  // (ready by the time the node is complete)
        } else {
          Real gp, inp;
          if (op & kLinkTree) {
            const uint32_t d = ((hdr >> kHdrDepthShift) & 63u) - 1u;
            gp = gstk[(size_t)d * 32];
            inp = istk[(size_t)d * 32];
          } else {
            const uint32_t p = op & kLinkIdxOut;
            gp = ga[(size_t)p * 32];
            inp = (op & kLinkOr) ? in_[(size_t)p * 32] : Real(0);
          }
          if (op & kLinkOr) {
            if (in_i > NI && gp > 0) g += gp * FNum<Real>::ex(in_i - inp);
          } else
            g += gp;
        }
        if (op & kOpLast) {
          if (hdr & kHdrPush) {  // an internal node: its children will ask for it
            const uint32_t d = (hdr >> kHdrDepthShift) & 63u;
            gstk[(size_t)d * 32] = g;
            istk[(size_t)d * 32] = in_i;
            ga[(size_t)jn * 32] = g;
          }
          const uint32_t lab = hdr & kHdrLabel;
          if (lab && g > 0) {
            if (hdr & kHdrHot)
              atomicAdd(A.hot + (size_t)replica * A.n_hot + hidx, (double)g);
            else
              atomicAdd(A.counts + lab, (double)g);
          }
          --jn;
        }
      }
    };
    uint32_t oa[kTileU];
    Real va[kTileU];
#pragma unroll
    for (int st = 0; st < kTileStages - 1; ++st) issue(st * kTileU);
    for (uint32_t s = 0; s < so; s += kTileU) {
      issue(s + (kTileStages - 1) * kTileU);   // (padded tail)
      f_cp_async_wait<kTileStages - 1>();  // chunk s/8 has landed
      ops_of(s, oa, va);
      process(oa, va);
    }
    f_cp_async_wait<0>();
  }
}

// ---------------------------------------------------------------------------------------------------
// Level-synchronous tiles (the throughput path for corpora of many small forests of ANY shape).
//
// A TILE is a run of consecutive forests whose nodes together fit in the CTA's shared memory (<= 32,768, 15-bit
// local ids).  The nodes of a tile are stored height-major ACROSS its forests: level 0 = the leaves of every
// forest of the tile, level 1 = ..., so one level is one contiguous slice of the arrays and the CTA's threads walk
// it with unit stride: label u32 + child/parent CSR offset u32 per node and pass, 16-bit local ids per link.  One
// value array lives in shared memory: after the inside pass it holds inside[node]; the outside pass visits the
// levels downwards and REPLACES a node's slot by the message its children need: gamma[node] (linear) for an AND
// node, ln gamma[node] - inside[node] for an OR node (a child of an OR parent adds exp(inside[child] + message)).
// Every gather of a child / parent value is a shared-memory read; global memory sees only the coalesced streams,
// read once per pass (DRAM traffic = the topology, no re-reads), and the rule weight / count tables (L2).
// Thread 0 requests the slices of the level `pf` steps ahead into L2 with cp.async.bulk.prefetch (TMA unit), so
// the dependent loads of a level (offsets, then links) pay L2 latency, not HBM latency; the per-thread loop keeps
// the next node's header loads in flight while the current node is reduced.  No divergence beyond the arity loop:
// lanes of a warp own consecutive nodes of the same level (k_forest_thread on an all-distinct corpus ran with 16
// of 32 lanes active and 2.7x the algorithmic DRAM traffic: profiles/round2_A_k_forest_thread.txt).
// ---------------------------------------------------------------------------------------------------
const uint32_t kLvlMaxLevels = 255, kLvlMaxNodes = 32768, kLvlOrParent = 0x8000u;
const int kLvlKids = 4, kLvlPars = 2;  // child / parent ids fetched ahead per node
struct __align__(16) LevelTile {
  uint64_t node_base;   // first entry of the tile in lt_label / lt_coff / lt_poff (n_nodes + 1 entries)
  uint64_t link_base;   // first link of the tile in lt_child / lt_par
  uint64_t lvl_base;    // 3 x (n_levels + 1) u32 in lt_lvl: node / child-link / parent-link offsets at the level boundaries
  uint32_t n_nodes, n_levels, n_forests;
  uint32_t forest_base; // first entry of the tile in lt_root / lt_forest
};
struct LevelArgs {
  const LevelTile* tiles;
  const uint32_t* label;      // inside pass: rule id (0 = OR)
  const uint32_t* label_out;  // outside pass: rule id, or bit 31 | replica row of a hot rule
  const uint32_t* coff;
  const uint32_t* poff;
  const uint16_t* child;
  const uint16_t* par;
  const uint32_t* lvl;
  const uint16_t* root;     // local id of each forest's root
  const uint32_t* forest;   // forest number within the batch (for ln_inside)
  const void* lnw;
  const uint32_t* hot_index;
  double* counts;
  double* hot;
  uint32_t n_hot;
  double* ln_inside;
  int pf;                   // L2 prefetch distance in levels (0 = off)
  uint32_t n_tiles;         // tiles of this launch (tiles points at the first)
  uint32_t cap;             // value slots of the largest tile
  uint32_t lvl_smem_off;    // byte offset of the level tables in dynamic shared memory (behind the values)
};
__device__ __forceinline__ void f_prefetch_l2(const void* base, size_t b0, size_t b1) {  // bytes [b0, b1) behind base
  const uintptr_t s = ((uintptr_t)base + b0) & ~(uintptr_t)15, e = ((uintptr_t)base + b1 + 15) & ~(uintptr_t)15;
  if (e > s) asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;\n" ::"l"((const void*)s), "r"((uint32_t)(e - s)) : "memory");
}
template <typename Real>
__device__ __forceinline__ Real f_log(Real x);
template <>
__device__ __forceinline__ float f_log<float>(float x) { return logf(x); }
template <>
__device__ __forceinline__ double f_log<double>(double x) { return log(x); }

// NTHR / MINB: threads per CTA and resident CTAs per SM the registers are capped for; U: nodes in flight per thread.
// (Measured and dropped: one WARP per small tile instead of a CTA -- no barriers, but levels of a few nodes leave most
// lanes idle: 13 of 32 lanes active, twice the warp instructions, 1.76 ms against 1.55 ms; profiles/round2_D_*.)
template <typename Real, int NTHR, int MINB, int U>
__global__ void __launch_bounds__(NTHR, MINB) k_forest_level(LevelArgs A) {
  extern __shared__ __align__(16) unsigned char smem_lv[];
  const uint32_t grp = blockIdx.x;
  Real* __restrict__ val = reinterpret_cast<Real*>(smem_lv);
  uint32_t* __restrict__ s_lvl = reinterpret_cast<uint32_t*>(smem_lv + A.lvl_smem_off);  // 3 x (levels + 1) words
  const LevelTile T = A.tiles[grp];
  const uint32_t tid = threadIdx.x, NT = blockDim.x, nl = T.n_levels;
  for (uint32_t k = tid; k < 3 * (nl + 1); k += NT) s_lvl[k] = __ldg(A.lvl + T.lvl_base + k);
  __syncthreads();
  auto sync = [&]() { __syncthreads(); };
  const uint32_t* __restrict__ s_node = s_lvl;
  const uint32_t* __restrict__ s_cl = s_lvl + (nl + 1);
  const uint32_t* __restrict__ s_pl = s_lvl + 2 * (nl + 1);
  const uint32_t* __restrict__ label = A.label + T.node_base;
  const uint32_t* __restrict__ label_o = A.label_out + T.node_base;
  const uint32_t* __restrict__ coff = A.coff + T.node_base;
  const uint32_t* __restrict__ poff = A.poff + T.node_base;
  const uint16_t* __restrict__ child = A.child + T.link_base;
  const uint16_t* __restrict__ par = A.par + T.link_base;
  const Real* __restrict__ lnw = (const Real*)A.lnw;
  const Real NI = FNum<Real>::ninf();
  const uint32_t pf = (uint32_t)A.pf;
  auto prefetch_in = [&](uint32_t L) {
    f_prefetch_l2(label, 4ull * s_node[L], 4ull * s_node[L + 1]);
    f_prefetch_l2(coff, 4ull * s_node[L], 4ull * s_node[L + 1] + 4);
    f_prefetch_l2(child, 2ull * s_cl[L], 2ull * s_cl[L + 1]);
  };
  auto prefetch_out = [&](uint32_t L) {
    f_prefetch_l2(label_o, 4ull * s_node[L], 4ull * s_node[L + 1]);
    f_prefetch_l2(poff, 4ull * s_node[L], 4ull * s_node[L + 1] + 4);
    f_prefetch_l2(par, 2ull * s_pl[L], 2ull * s_pl[L + 1]);
  };
  // ---- inside: ascending height (forest.hpp:636-697).  A thread keeps U nodes of the level in flight: all their
  // headers are loaded, then all their first kLvlKids child ids and rule weights, then they are reduced one by one --
  // with one node per thread and iteration the kernel ran at the latency of its dependent loads times the resident
  // threads (profiles/round2_B_k_forest_level.txt: 1.79 ms, DRAM 9 % busy, long-scoreboard + barrier stalls).
  if (tid == 0 && pf)
    for (uint32_t L = 0; L < pf && L < nl; ++L) prefetch_in(L);
  for (uint32_t L = 0; L < nl; ++L) {
    const uint32_t n1 = s_node[L + 1];
    if (tid == 0 && pf && L + pf < nl) prefetch_in(L + pf);
    if (L == 0) {  // height 0: leaves, inside = the rule weight
      for (uint32_t j0 = tid; j0 < n1; j0 += 2 * U * NT) {
        uint32_t lab[2 * U];
#pragma unroll
        for (int k = 0; k < 2 * U; ++k) {
          const uint32_t j = j0 + k * NT;
          lab[k] = j < n1 ? (__ldg(label + j) & ~kHotBit) : 0u;
        }
        Real wv[2 * U];
#pragma unroll
        for (int k = 0; k < 2 * U; ++k) wv[k] = __ldg(lnw + lab[k]);
#pragma unroll
        for (int k = 0; k < 2 * U; ++k) {
          const uint32_t j = j0 + k * NT;
          if (j < n1) val[j] = wv[k];
        }
      }
      sync();
      continue;
    }
    for (uint32_t j0 = s_node[L] + tid; j0 < n1; j0 += U * NT) {
      uint32_t lab[U], c0[U], c1[U];
#pragma unroll
      for (int k = 0; k < U; ++k) {
        const uint32_t j = j0 + k * NT;
        const bool ok = j < n1;
        lab[k] = ok ? (__ldg(label + j) & ~kHotBit) : 0u;
        c0[k] = ok ? __ldg(coff + j) : 0u;
        c1[k] = ok ? __ldg(coff + j + 1) : 0u;
      }
      uint32_t ch[U][kLvlKids];
      Real wv[U];
#pragma unroll
      for (int k = 0; k < U; ++k) {
#pragma unroll
        for (int q = 0; q < kLvlKids; ++q) ch[k][q] = (c0[k] + q < c1[k]) ? (uint32_t)__ldg(child + c0[k] + q) : 0u;
        wv[k] = __ldg(lnw + lab[k]);  // (entry 0 exists: rule ids start at 1)
      }
#pragma unroll
      for (int k = 0; k < U; ++k) {
        const uint32_t j = j0 + k * NT;
        if (j >= n1) continue;
        const uint32_t nc = c1[k] - c0[k];
        Real v;
        if (lab[k]) {  // AND: rule weight times the children
          v = wv[k];
#pragma unroll
          for (int q = 0; q < kLvlKids; ++q)
            if ((uint32_t)q < nc) v += val[ch[k][q]];
          for (uint32_t c = c0[k] + kLvlKids; c < c1[k]; ++c) v += val[__ldg(child + c)];
        } else {       // OR: the first child, then the others folded in the reference's order
          v = val[ch[k][0]];
#pragma unroll
          for (int q = 1; q < kLvlKids; ++q)
            if ((uint32_t)q < nc) v = ln_add_fast<Real>(v, val[ch[k][q]]);
          for (uint32_t c = c0[k] + kLvlKids; c < c1[k]; ++c) v = ln_add_fast<Real>(v, val[__ldg(child + c)]);
        }
        val[j] = v;
      }
    }
    sync();
  }
  for (uint32_t k = tid; k < T.n_forests; k += NT)
    A.ln_inside[__ldg(A.forest + T.forest_base + k)] = (double)val[__ldg(A.root + T.forest_base + k)];
  if (tid == 0 && pf)
    for (uint32_t d = 0; d < pf && d < nl; ++d) prefetch_out(nl - 1 - d);
  sync();
  // ---- outside as posteriors, descending height, pull over the parents (forest.hpp:439-491); a root (no parents) of a
  // zero-probability forest starts at 0, so that forest collects no counts (forest.hpp:447-451)
  const uint32_t replica = grp & (kHotCopies - 1);
  for (uint32_t L = nl; L-- > 0;) {
    const uint32_t n1 = s_node[L + 1];
    if (tid == 0 && pf && L >= pf) prefetch_out(L - pf);
    for (uint32_t j0 = s_node[L] + tid; j0 < n1; j0 += U * NT) {
      uint32_t lab[U], k0[U], k1[U];
#pragma unroll
      for (int k = 0; k < U; ++k) {
        const uint32_t j = j0 + k * NT;
        const bool ok = j < n1;
        lab[k] = ok ? __ldg(label_o + j) : 0u;
        k0[k] = ok ? __ldg(poff + j) : 0u;
        k1[k] = ok ? __ldg(poff + j + 1) : 0u;
      }
      uint32_t pa[U][kLvlPars];
#pragma unroll
      for (int k = 0; k < U; ++k) {
#pragma unroll
        for (int q = 0; q < kLvlPars; ++q) pa[k][q] = (k0[k] + q < k1[k]) ? (uint32_t)__ldg(par + k0[k] + q) : 0u;
      }
#pragma unroll
      for (int k = 0; k < U; ++k) {
        const uint32_t j = j0 + k * NT;
        if (j >= n1) continue;
        const Real in_i = val[j];
        const uint32_t np = k1[k] - k0[k];
        Real g;
        if (np == 0)
          g = in_i > NI ? Real(1) : Real(0);
        else {
          g = 0;
          auto add = [&](uint32_t e) {
            const Real m = val[e & (kLvlOrParent - 1)];
            if (e & kLvlOrParent) {  // OR parent: this alternative's share, m = ln gamma[p] - inside[p]
              if (in_i > NI) g += FNum<Real>::ex(in_i + m);
            } else
              g += m;                // AND parent: every child is used whenever the parent is
          };
#pragma unroll
          for (int q = 0; q < kLvlPars; ++q)
            if ((uint32_t)q < np) add(pa[k][q]);
          for (uint32_t kk = k0[k] + kLvlPars; kk < k1[k]; ++kk) add(__ldg(par + kk));
        }
        if (lab[k]) {  // an AND node (the label of a hot rule is bit 31 | its replica row, never 0)
          if (g > 0) {
            if (lab[k] & kHotBit)
              atomicAdd(A.hot + (size_t)replica * A.n_hot + (lab[k] & ~kHotBit), (double)g);
            else
              atomicAdd(A.counts + lab[k], (double)g);
          }
          if (L) val[j] = g;
        } else if (L)
          val[j] = (g > 0 && in_i > NI) ? f_log<Real>(g) - in_i : NI;
      }
    }
    sync();
  }
}

// mark hot rules in the headers of the outside streams (bit 22); idempotent
__global__ void k_forest_mark_hot_ops(uint64_t n, uint32_t* __restrict__ ops, const uint32_t* __restrict__ hot_index) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint32_t op = ops[i];
  if (op == kOpNop || !(op & kHdr)) return;
  const uint32_t lab = op & kHdrLabel;
  ops[i] = (lab && hot_index[lab] != 0xFFFFFFFFu) ? (op | kHdrHot) : (op & ~kHdrHot);
}

// mark hot rules in the node labels (bit 31); idempotent
__global__ void k_forest_mark_hot(uint64_t n, uint32_t* __restrict__ label, const uint32_t* __restrict__ hot_index) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint32_t lab = label[i] & ~kHotBit;
  label[i] = (lab && hot_index[lab] != 0xFFFFFFFFu) ? (lab | kHotBit) : lab;
}
// level tiles: the outside pass's label stream carries the replica ROW of a hot rule instead of its id (bit 31 set), so
// the count of a hot rule needs no lookup; derived from the inside pass's labels whenever the hot set changes
__global__ void k_forest_label_out(uint64_t n, const uint32_t* __restrict__ label, const uint32_t* __restrict__ hot_index,
                                   uint32_t* __restrict__ out) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint32_t lab = label[i] & ~kHotBit;
  const uint32_t h = lab ? hot_index[lab] : 0xFFFFFFFFu;
  out[i] = h != 0xFFFFFFFFu ? (h | kHotBit) : lab;
}
__global__ void k_forest_fold(uint32_t n_hot, const uint32_t* __restrict__ hot_rule, const double* __restrict__ hot,
                              double* __restrict__ counts) {
  const uint32_t h = blockIdx.x * blockDim.x + threadIdx.x;
  if (h >= n_hot) return;
  double s = 0;
#pragma unroll 8
  for (int k = 0; k < kHotCopies; ++k) s += hot[(size_t)k * n_hot + h];
  if (s != 0.) atomicAdd(&counts[hot_rule[h]], s);
}
// sum of ln inside over non-zero forests (forest-em.hpp:519-527): one block, fixed order => deterministic
// stage 1: kSumBlocks blocks, block b sums the fixed slice b of the forests into partial[2b..2b+1]
const int kSumBlocks = 128;
__global__ void k_forest_sum_partial(const double* __restrict__ ln_inside, uint64_t n, double* __restrict__ partial) {
  __shared__ double s_sum[256];
  __shared__ double s_zero[256];
  const uint64_t per = (n + gridDim.x - 1) / gridDim.x;
  const uint64_t b = blockIdx.x * per, e = b + per < n ? b + per : n;
  double s = 0, z = 0;
  for (uint64_t i = b + threadIdx.x; i < e; i += blockDim.x) {
    const double v = ln_inside[i];
    if (v > -CUDART_INF)
      s += v;
    else
      z += 1;
  }
  s_sum[threadIdx.x] = s;
  s_zero[threadIdx.x] = z;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if ((int)threadIdx.x < o) {
      s_sum[threadIdx.x] += s_sum[threadIdx.x + o];
      s_zero[threadIdx.x] += s_zero[threadIdx.x + o];
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    partial[2 * blockIdx.x] = s_sum[0];
    partial[2 * blockIdx.x + 1] = s_zero[0];
  }
}
// stage 2 (one block): fold the partials (pairs: sum, zeros) in a fixed order
__global__ void k_forest_sum(const double* __restrict__ ln_inside, uint64_t n, double* __restrict__ scal, uint64_t n_forests) {
  __shared__ double s_sum[256];
  __shared__ double s_zero[256];
  double s = 0, z = 0;
  for (uint64_t i = threadIdx.x; i < n; i += blockDim.x) {
    s += ln_inside[2 * i];
    z += ln_inside[2 * i + 1];
  }
  s_sum[threadIdx.x] = s;
  s_zero[threadIdx.x] = z;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if ((int)threadIdx.x < o) {
      s_sum[threadIdx.x] += s_sum[threadIdx.x + o];
      s_zero[threadIdx.x] += s_zero[threadIdx.x + o];
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    scal[0] += s_sum[0];
    scal[1] += s_zero[0];
    scal[2] += (double)n_forests;
  }
}
template <typename Real>
__global__ void k_forest_cast_w(uint64_t n, const double* __restrict__ ln_w, Real* __restrict__ out) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = (Real)ln_w[i];
}
// NormalizeGroups::operator()(Group&) (normalize.hpp:123-164): one warp per group.
// src = counts + prior (linear) or exp(ln_w) when counts == nullptr (normalize in place).
__global__ void k_forest_norm(uint64_t n_groups, const uint64_t* __restrict__ goff, const uint64_t* __restrict__ gmem,
                              const double* __restrict__ counts, double prior, double add_k, int zero_mode,
                              double* __restrict__ ln_w, double* __restrict__ gdiff, uint64_t* __restrict__ gidx) {
  const uint64_t g = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (g >= n_groups) return;
  const uint64_t b = goff[g], e = goff[g + 1];
  double sum = 0;
  for (uint64_t k = b + lane; k < e; k += 32) {
    const uint64_t r = gmem[k];
    sum += counts ? counts[r] + prior : exp(ln_w[r]);
  }
  for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
  double best = -1;
  uint64_t best_k = ~0ull;
  if (sum > 0) {
    const double ln_den = log(sum + add_k);
    for (uint64_t k = b + lane; k < e; k += 32) {
      const uint64_t r = gmem[k];
      const double c = counts ? counts[r] + prior : exp(ln_w[r]);
      const double prev = ln_w[r];
      const double nw = c > 0 ? log(c) - ln_den : -CUDART_INF;
      ln_w[r] = nw;
      const double diff = fabs(exp(nw) - exp(prev));
      if (diff > best) {
        best = diff;
        best_k = k;
      }
    }
  } else if (zero_mode != CML_FOREST_SKIP) {
    const double setto = zero_mode == CML_FOREST_UNIFORM ? -log((double)(e - b)) : -CUDART_INF;
    for (uint64_t k = b + lane; k < e; k += 32) {
      const uint64_t r = gmem[k];
      const double diff = fabs(exp(setto) - exp(ln_w[r]));
      ln_w[r] = setto;
      if (diff > best) {
        best = diff;
        best_k = k;
      }
    }
  }
  // first maximum in member order (the reference keeps the first strictly larger difference)
  for (int o = 16; o > 0; o >>= 1) {
    const double ob = __shfl_xor_sync(0xffffffffu, best, o);
    const uint64_t ok = __shfl_xor_sync(0xffffffffu, best_k, o);
    if (ob > best || (ob == best && ok < best_k)) {
      best = ob;
      best_k = ok;
    }
  }
  if (lane == 0) {
    gdiff[g] = best;
    gidx[g] = best_k;
  }
}
// final reduction over groups: largest difference, ties -> first group
__global__ void k_forest_maxdiff(uint64_t n_groups, const double* __restrict__ gdiff, const uint64_t* __restrict__ gidx,
                                 const uint64_t* __restrict__ gmem, double* __restrict__ out_diff,
                                 unsigned long long* __restrict__ out_rule) {
  __shared__ double s_d[1024];
  __shared__ uint64_t s_g[1024];
  double best = 0;  // maxdiff starts at zero and needs a strictly larger difference (normalize.hpp:258)
  uint64_t bg = ~0ull;
  // one block of 1024 threads, 4 loads in flight per thread (a 256-thread block walking 40 k groups one dependent load at
  // a time was most of the M-step's time)
  for (uint64_t g0 = threadIdx.x; g0 < n_groups; g0 += 4ull * blockDim.x) {
    double d[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const uint64_t g = g0 + (uint64_t)k * blockDim.x;
      d[k] = g < n_groups ? gdiff[g] : 0.;
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const uint64_t g = g0 + (uint64_t)k * blockDim.x;
      if (g < n_groups && (d[k] > best || (d[k] == best && d[k] > 0 && g < bg))) {
        best = d[k];
        bg = g;
      }
    }
  }
  s_d[threadIdx.x] = best;
  s_g[threadIdx.x] = bg;
  __syncthreads();
  for (int o = (int)blockDim.x / 2; o > 0; o >>= 1) {
    if ((int)threadIdx.x < o) {
      const double d = s_d[threadIdx.x + o];
      const uint64_t g = s_g[threadIdx.x + o];
      if (d > s_d[threadIdx.x] || (d == s_d[threadIdx.x] && g < s_g[threadIdx.x])) {
        s_d[threadIdx.x] = d;
        s_g[threadIdx.x] = g;
      }
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    *out_diff = s_d[0];
    *out_rule = s_g[0] == ~0ull ? 0ull : (unsigned long long)gmem[gidx[s_g[0]]];
  }
}

struct ForestBatch {
  uint64_t n_forests = 0, n_nodes = 0, n_links = 0, n_hyperedges = 0, max_nodes = 0;
  DevArray<ForestDesc> desc;
  DevArray<uint32_t> label, child_off, par_off, child, par, lvl_off, list;
  DevArray<double> ln_inside;
  uint32_t cls_begin[kNWarpCls + 2] = {0};  // warp classes, then the CTA class
  DevArray<unsigned char> scratch;
  uint64_t scratch_stride = 0;
  uint32_t cta_grid = 0;
  // thread-per-forest tiles
  uint32_t n_tiles = 0;
  uint64_t t_forests = 0, t_steps = 0, t_rows = 0;  // forests in tiles; real (unpadded) steps; padded rows * 32
  DevArray<TileDesc> tiles;
  DevArray<uint32_t> t_ops_in, t_ops_out;
  uint32_t t_stack_rows = 2;  // shared-memory rows per lane for the value / path stacks
  DevArray<unsigned char> t_in, t_ga, t_vout;
  // level-synchronous tiles
  uint32_t n_ltiles = 0, lt_max_nodes = 0, lt_max_levels = 0;  // level tiles; nodes / levels of the largest tile
  uint32_t n_stiles = 0, lt_small_nodes = 0;  // the first n_stiles tiles are SMALL tiles (largest: lt_small_nodes nodes)
  uint64_t lt_forests = 0, lt_nodes = 0, lt_links = 0;
  DevArray<LevelTile> ltiles;
  DevArray<uint32_t> lt_label, lt_label_out, lt_coff, lt_poff, lt_lvl, lt_forest;
  DevArray<uint16_t> lt_child, lt_par, lt_root;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  uint32_t n_kernels = 0;
  ~ForestBatch() {
    if (ev0) cudaEventDestroy(ev0);
    if (ev1) cudaEventDestroy(ev1);
  }
};

}  // namespace

struct cml_forests {
  int device = 0, precision = 32;
  cudaStream_t stream = nullptr;
  bool own_stream = false;
  int sm_count = CML_SM_COUNT_FALLBACK;
  size_t smem_optin = 0;
  std::string err;
  uint64_t launches = 0;
  bool have_rules = false, have_params = false, hot_dirty = true, pending = false;
  int layout = CML_FOREST_LAYOUT_AUTO;
  uint64_t rulespace = 0, n_groups = 0;
  DevArray<uint64_t> group_off, group_members;
  DevArray<double> ln_w, reduce, gdiff, out_diff, sum_partial;
  DevArray<uint64_t> gidx;
  DevArray<unsigned long long> out_rule;
  DevArray<unsigned char> w_real;
  std::vector<uint64_t> rule_occ;
  DevArray<uint32_t> hot_index, hot_rule;
  DevArray<double> hot;
  uint32_t n_hot = 0;
  std::vector<std::unique_ptr<ForestBatch>> batches;
  // --crp Gibbs sampling (cml_forests_gibbs_*): the forests in the reference representation, CRP state, samples
  bool have_gibbs = false;
  uint64_t g_forests = 0, g_nodes = 0, g_cap = 0;
  uint32_t g_norms = 0;
  int g_cur = 0;
  DevArray<uint64_t> g_node_off, g_samp_base;
  DevArray<uint32_t> g_next, g_label, g_norm, g_sample[2], g_len[2];
  DevArray<uint8_t> g_backref;
  DevArray<double> g_prior, g_count, g_cum, g_normsum, g_ins;
  DevArray<int> g_err;
  void* comm = nullptr;  // ncclComm_t of this rank (cml_forests_comm_init_rank), null on a single GPU
  int comm_size = 1;
  uint64_t collectives = 0;
  // cml_forests_kbest: scratch budget of one chunk, and the last call's scratch / chunks / kernel time
  uint64_t kbest_scratch_mb = 4096, kbest_scratch = 0, kbest_chunks = 0;
  float kbest_ms = 0;
  // cml_forests_sample (chunks under the same budget): the last call's scratch / chunks / kernel time
  uint64_t sample_scratch = 0, sample_chunks = 0;
  float sample_ms = 0;
};
// cml_comm.cu
int cml_nccl_init_rank(void** comm, int n_ranks, int rank, const unsigned char* id, std::string& err);
int cml_nccl_allreduce(void* comm, double* p, uint64_t count, cudaStream_t s, std::string& err);
void cml_nccl_destroy(void* comm);

#define ctx f
#define F_REQUIRE(cond, code, msg) \
  do {                             \
    if (!(cond)) {                 \
      f->err = (msg);              \
      return (code);               \
    }                              \
  } while (0)

static thread_local std::string g_forest_create_err;
static inline unsigned f_cdiv(uint64_t a, uint64_t b) { return (unsigned)((a + b - 1) / b); }

extern "C" int cml_forests_create(cml_forests** out, int device, int precision) {
  if (!out || (precision != 32 && precision != 64)) {
    g_forest_create_err = "cml_forests_create: precision must be 32 or 64";
    return CML_ERR_ARG;
  }
  *out = nullptr;
  int n_dev = 0;
  if (cudaGetDeviceCount(&n_dev) != cudaSuccess || device < 0 || device >= n_dev) {
    g_forest_create_err = "cml_forests_create: no usable CUDA device " + std::to_string(device) +
                          " (carmel_b200 has no CPU fallback)";
    return CML_ERR_CUDA;
  }
  std::unique_ptr<cml_forests> f(new cml_forests());
  f->device = device;
  f->precision = precision;
  if (cudaSetDevice(device) != cudaSuccess || cudaStreamCreateWithFlags(&f->stream, cudaStreamNonBlocking) != cudaSuccess) {
    g_forest_create_err = "cml_forests_create: cannot initialise the device";
    return CML_ERR_CUDA;
  }
  f->own_stream = true;
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) == cudaSuccess) {
    f->sm_count = prop.multiProcessorCount;
    f->smem_optin = prop.sharedMemPerBlockOptin;
  }
  *out = f.release();
  return CML_OK;
}
extern "C" void cml_forests_destroy(cml_forests* f) {
  if (!f) return;
  cudaSetDevice(f->device);
  cudaStreamSynchronize(f->stream);
  f->batches.clear();
  cml_nccl_destroy(f->comm);
  if (f->own_stream) cudaStreamDestroy(f->stream);
  delete f;
}
// the per-iteration all-reduce of [rule counts | sum ln inside | n_zero | n_forests] (north_star (4)); same rendezvous
// token scheme as cml_comm_init_rank
extern "C" int cml_forests_comm_init_rank(cml_forests* f, int n_ranks, int rank, const unsigned char id[CML_COMM_ID_BYTES]) {
  if (!f || !id || n_ranks < 1 || rank < 0 || rank >= n_ranks) return CML_ERR_ARG;
  cudaSetDevice(f->device);
  cml_nccl_destroy(f->comm);
  f->comm = nullptr;
  const int r = cml_nccl_init_rank(&f->comm, n_ranks, rank, id, f->err);
  if (r) return r;
  f->comm_size = n_ranks;
  return CML_OK;
}
extern "C" int cml_forests_allreduce_counts(cml_forests* f) {
  if (!f) return CML_ERR_ARG;
  if (!f->comm || f->comm_size <= 1) return CML_OK;
  cudaSetDevice(f->device);
  ++f->collectives;
  return cml_nccl_allreduce(f->comm, f->reduce.p, f->rulespace + 3, f->stream, f->err);
}
extern "C" int cml_forests_synchronize(cml_forests* f) {
  if (!f) return CML_ERR_ARG;
  cudaSetDevice(f->device);
  CML_CUDA(cudaStreamSynchronize(f->stream));
  return CML_OK;
}
extern "C" const char* cml_forests_last_error(cml_forests* f) { return f ? f->err.c_str() : g_forest_create_err.c_str(); }
extern "C" int cml_forests_set_stream(cml_forests* f, void* s) {
  if (!f) return CML_ERR_ARG;
  CML_CUDA(cudaStreamSynchronize(f->stream));
  if (f->own_stream) cudaStreamDestroy(f->stream);
  f->stream = (cudaStream_t)s;
  f->own_stream = false;
  return CML_OK;
}
extern "C" uint64_t cml_forests_launch_count(cml_forests* f) { return f ? f->launches : 0; }
extern "C" int cml_forests_set_layout(cml_forests* f, int layout) {
  if (!f) return CML_ERR_ARG;
  F_REQUIRE(layout >= CML_FOREST_LAYOUT_AUTO && layout <= CML_FOREST_LAYOUT_LEVEL, CML_ERR_ARG, "cml_forests_set_layout: unknown layout");
  f->layout = layout;
  return CML_OK;
}
extern "C" int cml_forests_layout_stats(cml_forests* f, uint64_t* tile_forests, uint64_t* tiles, uint64_t* steps, uint64_t* padded_steps,
                                        uint64_t* padded_rows) {
  if (!f) return CML_ERR_ARG;
  uint64_t a = 0, b = 0, c = 0, d = 0, e = 0;
  for (auto const& bt : f->batches) {
    a += bt->t_forests;
    b += bt->n_tiles;
    c += bt->t_steps;
    d += bt->t_ops_in.n * (bt->n_tiles ? 1 : 0) + bt->t_ops_out.n * (bt->n_tiles ? 1 : 0);
    e += bt->t_rows;
  }
  if (tile_forests) *tile_forests = a;
  if (tiles) *tiles = b;
  if (steps) *steps = c;
  if (padded_steps) *padded_steps = d;
  if (padded_rows) *padded_rows = e;
  return CML_OK;
}

extern "C" int cml_forests_level_stats(cml_forests* f, uint64_t* forests, uint64_t* tiles, uint64_t* nodes, uint64_t* links,
                                       uint64_t* max_tile_nodes, uint64_t* small_tiles) {
  if (!f) return CML_ERR_ARG;
  uint64_t a = 0, b = 0, c = 0, d = 0, e = 0, w = 0;
  for (auto const& bt : f->batches) {
    a += bt->lt_forests;
    b += bt->n_ltiles;
    c += bt->lt_nodes;
    d += bt->lt_links;
    e = std::max<uint64_t>(e, std::max(bt->lt_max_nodes, bt->lt_small_nodes));
    w += bt->n_stiles;
  }
  if (small_tiles) *small_tiles = w;
  if (forests) *forests = a;
  if (tiles) *tiles = b;
  if (nodes) *nodes = c;
  if (links) *links = d;
  if (max_tile_nodes) *max_tile_nodes = e;
  return CML_OK;
}

extern "C" int cml_forests_set_rules(cml_forests* f, uint64_t rulespace, uint64_t n_groups, const uint64_t* group_off,
                                     const uint64_t* group_members) {
  if (!f) return CML_ERR_ARG;
  F_REQUIRE(rulespace >= 1 && rulespace < 0x7fffffffull, CML_ERR_ARG, "cml_forests_set_rules: rulespace out of range");
  F_REQUIRE(f->batches.empty(), CML_ERR_STATE, "cml_forests_set_rules: forests already added");
  F_REQUIRE(n_groups == 0 || (group_off && group_members), CML_ERR_ARG, "cml_forests_set_rules: null groups");
  std::vector<char> seen(rulespace, 0);
  for (uint64_t g = 0; g < n_groups; ++g) {
    F_REQUIRE(group_off[g] <= group_off[g + 1], CML_ERR_ARG, "cml_forests_set_rules: group offsets not monotone");
    for (uint64_t k = group_off[g]; k < group_off[g + 1]; ++k)
      F_REQUIRE(group_members[k] < rulespace, CML_ERR_ARG, "cml_forests_set_rules: group member beyond rulespace");
  }
  CML_CUDA(cudaSetDevice(f->device));
  const uint64_t n_mem = n_groups ? group_off[n_groups] : 0;
  static const uint64_t zero_off[1] = {0};
  CML_CUDA(f->group_off.upload(n_groups ? group_off : zero_off, n_groups + 1, f->stream));
  CML_CUDA(f->group_members.upload(group_members, n_mem, f->stream));
  CML_CUDA(f->ln_w.alloc(rulespace));
  CML_CUDA(f->w_real.alloc(rulespace * (f->precision == 64 ? 8 : 4)));
  CML_CUDA(f->reduce.alloc(rulespace + 3));
  CML_CUDA(cudaMemsetAsync(f->reduce.p, 0, (rulespace + 3) * sizeof(double), f->stream));
  CML_CUDA(f->gdiff.alloc(std::max<uint64_t>(1, n_groups)));
  CML_CUDA(f->gidx.alloc(std::max<uint64_t>(1, n_groups)));
  CML_CUDA(f->out_diff.alloc(1));
  CML_CUDA(f->out_rule.alloc(1));
  CML_CUDA(cudaStreamSynchronize(f->stream));
  f->rulespace = rulespace;
  f->n_groups = n_groups;
  f->rule_occ.assign(rulespace, 0);
  f->have_rules = true;
  f->have_params = false;
  f->hot_dirty = true;
  return CML_OK;
}
extern "C" int cml_forests_set_params(cml_forests* f, const double* ln_w) {
  if (!f || !ln_w) return CML_ERR_ARG;
  F_REQUIRE(f->have_rules, CML_ERR_STATE, "cml_forests_set_params before cml_forests_set_rules");
  CML_CUDA(cudaSetDevice(f->device));
  CML_CUDA(cudaMemcpyAsync(f->ln_w.p, ln_w, f->rulespace * sizeof(double), cudaMemcpyHostToDevice, f->stream));
  CML_CUDA(cudaStreamSynchronize(f->stream));
  f->have_params = true;
  return CML_OK;
}
extern "C" int cml_forests_get_params(cml_forests* f, double* ln_w) {
  if (!f || !ln_w) return CML_ERR_ARG;
  F_REQUIRE(f->have_params, CML_ERR_STATE, "cml_forests_get_params before cml_forests_set_params");
  CML_CUDA(cudaSetDevice(f->device));
  CML_CUDA(cudaMemcpyAsync(ln_w, f->ln_w.p, f->rulespace * sizeof(double), cudaMemcpyDeviceToHost, f->stream));
  CML_CUDA(cudaStreamSynchronize(f->stream));
  return CML_OK;
}

// ---------------------------------------------------------------------------------------------------
// host-side layout: pre-order node arrays -> height-sorted hyperedge CSRs
// ---------------------------------------------------------------------------------------------------
namespace {
struct FlatForest {
  uint32_t n_real = 0, n_levels = 0, n_leaves = 0;
  uint64_t n_links = 0, n_he = 0;
  int error = 0;  // 1 malformed, 2 cycle, 3 rule id out of range
};
struct ForestScratch {
  std::vector<uint32_t> height, order, newid, stack, it, cnt, post, tpar, depth, sim, kids, npar;
  std::vector<char> color;
};
// pass 1: validate, heights, counts.  `real_of[i]` for pre-order node i = i or the target of a back reference.
void forest_pass1(uint32_t n, const uint32_t* next, const uint32_t* label, const uint8_t* backref, uint64_t rulespace,
                  ForestScratch& S, FlatForest& ff) {
  ff = FlatForest();
  if (n == 0 || backref[0] || next[0] != n) {
    ff.error = 1;
    return;
  }
  for (uint32_t i = 0; i < n; ++i) {
    if (next[i] <= i || next[i] > n) {
      ff.error = 1;
      return;
    }
    if (backref[i]) {
      if (label[i] >= n || backref[label[i]] || next[i] != i + 1) {
        ff.error = 1;
        return;
      }
    } else {
      if (label[i] >= rulespace) {
        ff.error = 3;
        return;
      }
      if (label[i] == 0 && next[i] == i + 1) {  // OR without children
        ff.error = 1;
        return;
      }
    }
  }
  // children of real node p: b = p+1; while b < next[p]: (backref ? label[b] : b); b = next[b]
  S.height.assign(n, 0);
  S.color.assign(n, 0);
  S.stack.clear();
  S.post.clear();     // DFS post-order of the real nodes (children before parents, the root last)
  S.it.assign(n, 0);  // resume position (pre-order index of the next child to look at)
  S.stack.push_back(0);
  S.color[0] = 1;
  S.it[0] = 1;
  while (!S.stack.empty()) {
    const uint32_t p = S.stack.back();
    uint32_t b = S.it[p];
    if (b < next[p]) {
      if (next[b] > next[p]) {  // child sticks out of its parent
        ff.error = 1;
        return;
      }
      S.it[p] = next[b];
      const uint32_t c = backref[b] ? label[b] : b;
      ++ff.n_links;
      if (S.color[c] == 1) {
        ff.error = 2;
        return;
      }
      if (S.color[c] == 0) {
        S.color[c] = 1;
        S.it[c] = c + 1;
        S.stack.push_back(c);
      }
    } else {
      uint32_t h = 0;
      for (uint32_t q = p + 1; q < next[p]; q = next[q]) {
        const uint32_t c = backref[q] ? label[q] : q;
        h = std::max(h, S.height[c] + 1);
      }
      S.height[p] = h;
      S.color[p] = 2;
      S.post.push_back(p);
      if (next[p] == p + 1) ++ff.n_leaves;
      S.stack.pop_back();
    }
  }
  uint32_t n_real = 0, maxh = 0;
  for (uint32_t i = 0; i < n; ++i)
    if (!backref[i]) {
      if (S.color[i] != 2) {  // a shared definition that is never reached cannot happen in pre-order text
        ff.error = 1;
        return;
      }
      ++n_real;
      maxh = std::max(maxh, S.height[i]);
      if (label[i]) ++ff.n_he;
    }
  ff.n_real = n_real;
  ff.n_levels = maxh + 1;
}
}  // namespace

extern "C" int cml_forests_add(cml_forests* f, const cml_forest_batch* b) {
  if (!f || !b) return CML_ERR_ARG;
  F_REQUIRE(f->have_rules, CML_ERR_STATE, "cml_forests_add before cml_forests_set_rules");
  F_REQUIRE(!f->pending, CML_ERR_STATE, "cml_forests_add while an estimate is pending");
  F_REQUIRE(b->n_forests == 0 || (b->node_off && b->next && b->label && b->backref), CML_ERR_ARG, "cml_forests_add: null array");
  if (b->n_forests == 0) return CML_OK;
  const uint64_t nf = b->n_forests;
  for (uint64_t i = 0; i < nf; ++i) {
    F_REQUIRE(b->node_off[i] < b->node_off[i + 1], CML_ERR_ARG, "cml_forests_add: empty forest");
    F_REQUIRE(b->node_off[i + 1] - b->node_off[i] < 0x7fffffffull, CML_ERR_ARG, "cml_forests_add: forest too large");
  }
  CML_CUDA(cudaSetDevice(f->device));
  unsigned nt = std::max(1u, std::min(32u, std::thread::hardware_concurrency()));
  if (nf < 64) nt = 1;
  std::vector<FlatForest> ff(nf);
  {
    std::atomic<uint64_t> nextf(0);
    auto work = [&]() {
      ForestScratch S;
      for (;;) {
        const uint64_t i0 = nextf.fetch_add(64);
        if (i0 >= nf) break;
        for (uint64_t i = i0; i < std::min(nf, i0 + 64); ++i) {
          const uint64_t o = b->node_off[i];
          forest_pass1((uint32_t)(b->node_off[i + 1] - o), b->next + o, b->label + o, b->backref + o, f->rulespace, S, ff[i]);
        }
      }
    };
    std::vector<std::thread> th;
    for (unsigned t = 1; t < nt; ++t) th.emplace_back(work);
    work();
    for (auto& t : th) t.join();
  }
  std::unique_ptr<ForestBatch> bt(new ForestBatch());
  std::vector<uint64_t> node_base(nf + 1, 0), link_base(nf + 1, 0), lvl_base(nf + 1, 0);
  for (uint64_t i = 0; i < nf; ++i) {
    if (ff[i].error) {
      f->err = "cml_forests_add: forest " + std::to_string(i) +
               (ff[i].error == 2 ? " has a cyclic back reference" : ff[i].error == 3 ? " uses a rule id beyond rulespace" : " is malformed");
      return ff[i].error == 2 ? CML_ERR_CYCLE : CML_ERR_ARG;
    }
    bt->n_nodes += ff[i].n_real;
    bt->n_links += ff[i].n_links;
    bt->n_hyperedges += ff[i].n_he;
    bt->max_nodes = std::max<uint64_t>(bt->max_nodes, ff[i].n_real);
  }
  // layout family per forest: thread-per-forest tiles for corpora of many small forests, else warp / CTA per forest
  std::vector<char> in_tile(nf, 0), in_level(nf, 0);
  const size_t real_bytes = f->precision == 64 ? 8 : 4;
  // level-synchronous tiles (k_forest_level): runs of consecutive forests whose nodes fit in a CTA's shared memory
  std::vector<uint32_t> lv_forests;           // forests in level tiles, tile-major (corpus order)
  std::vector<uint32_t> lv_first;             // per tile: first entry in lv_forests (+ sentinel)
  // two tile classes: SMALL tiles for the launch shape 128 threads x 16 CTAs per SM (full occupancy, 16 independent
  // barrier domains per SM: measured best, profiles/round2_F_*), LARGE tiles (512 x 2) for forests that do not fit a
  // small tile's shared memory.  Tiles [0, lv_n_small) are small.
  uint32_t lv_n_small = 0;
  {
    uint64_t min_forests = 256, kb_small = 12, kb_large = 100;  // (16 x (12 KB + tables + 1 KB reserved) fit one SM)
    if (const char* e = getenv("CML_FOREST_LEVEL_MIN_FORESTS")) min_forests = std::strtoull(e, nullptr, 10);
    if (const char* e = getenv("CML_FOREST_LEVEL_SMEM_KB")) kb_small = std::strtoull(e, nullptr, 10);  // (0: no small tiles)
    if (const char* e = getenv("CML_FOREST_LEVEL_LARGE_KB")) kb_large = std::strtoull(e, nullptr, 10);
    kb_large = std::min<uint64_t>(kb_large, f->smem_optin ? (f->smem_optin - 4096) / 1024 : 100);
    kb_small = std::min(kb_small, kb_large);
    uint32_t max_lev = 1;  // the level tables of a tile (3 x (levels + 1) words) share the CTA's shared memory
    for (uint64_t i = 0; i < nf; ++i)
      if (ff[i].n_levels <= kLvlMaxLevels) max_lev = std::max(max_lev, ff[i].n_levels);
    const uint64_t lvl_bytes = (12ull * (max_lev + 1) + 15) & ~15ull;
    auto cap_of = [&](uint64_t kb) {
      return std::min<uint64_t>(kLvlMaxNodes, (kb * 1024 - std::min<uint64_t>(lvl_bytes, kb * 512)) / real_bytes);
    };
    const uint64_t cap_small = kb_small ? cap_of(kb_small) : 0, cap = cap_of(kb_large);
    uint64_t cand = 0;
    for (uint64_t i = 0; i < nf; ++i) cand += ff[i].n_real <= cap && ff[i].n_levels <= kLvlMaxLevels;
    const bool use = f->layout == CML_FOREST_LAYOUT_LEVEL || (f->layout == CML_FOREST_LAYOUT_AUTO && cand >= min_forests);
    if (use && cand) {
      auto eligible = [&](uint64_t i) { return ff[i].n_real <= cap && ff[i].n_levels <= kLvlMaxLevels; };
      auto pack = [&](uint64_t lo, uint64_t hi, uint64_t tile_cap) {  // forests of lo < n_real <= hi, corpus order
        uint64_t nodes = 0;
        for (uint64_t i = 0; i < nf; ++i)
          if (eligible(i) && ff[i].n_real > lo && ff[i].n_real <= hi) nodes += ff[i].n_real;
        // small corpora: smaller tiles so that there are a few CTAs per SM
        uint64_t target = std::max<uint64_t>(1024, nodes / (8ull * (uint64_t)f->sm_count));
        if (const char* e = getenv("CML_FOREST_LEVEL_TILE_NODES")) target = std::strtoull(e, nullptr, 10);
        target = std::min(target, tile_cap);
        uint64_t cur = 0;
        bool first = true;
        for (uint64_t i = 0; i < nf; ++i) {
          if (!eligible(i) || !(ff[i].n_real > lo && ff[i].n_real <= hi)) continue;
          in_level[i] = 1;
          if (first || cur + ff[i].n_real > std::max<uint64_t>(target, ff[i].n_real)) {
            lv_first.push_back((uint32_t)lv_forests.size());
            cur = 0;
            first = false;
          }
          cur += ff[i].n_real;
          lv_forests.push_back((uint32_t)i);
        }
      };
      if (cap_small) pack(0, cap_small, cap_small);
      lv_n_small = (uint32_t)lv_first.size();
      pack(cap_small, cap, cap);
      lv_first.push_back((uint32_t)lv_forests.size());
    }
  }
  {
    uint64_t min_forests = 8192, max_nodes = 16384;
    if (const char* e = getenv("CML_FOREST_TILE_MIN_FORESTS")) min_forests = std::strtoull(e, nullptr, 10);
    if (const char* e = getenv("CML_FOREST_TILE_MAX_NODES")) max_nodes = std::strtoull(e, nullptr, 10);
    uint64_t cand = 0;
    for (uint64_t i = 0; i < nf; ++i) cand += !in_level[i] && ff[i].n_real <= max_nodes;
    const bool labels_fit = f->rulespace <= (uint64_t)kHdrLabel + 1;  // the stream headers carry 22-bit rule ids
    const bool use = labels_fit &&
                     (f->layout == CML_FOREST_LAYOUT_THREAD || (f->layout == CML_FOREST_LAYOUT_AUTO && cand >= min_forests));
    if (use)
      for (uint64_t i = 0; i < nf; ++i) in_tile[i] = !in_level[i] && (ff[i].n_real <= max_nodes || f->layout == CML_FOREST_LAYOUT_THREAD);
  }
  for (uint64_t i = 0; i < nf; ++i) {
    const bool g = !in_tile[i] && !in_level[i];
    node_base[i + 1] = node_base[i] + (g ? ff[i].n_real + 1 : 0);
    link_base[i + 1] = link_base[i] + (g ? ff[i].n_links : 0);
    lvl_base[i + 1] = lvl_base[i] + (g ? ff[i].n_levels + 1 : 0);
  }
  bt->n_forests = nf;
  std::vector<ForestDesc> desc(nf);
  std::vector<uint32_t> h_label(node_base[nf]), h_coff(node_base[nf]), h_poff(node_base[nf]), h_child(std::max<uint64_t>(1, link_base[nf])),
      h_par(std::max<uint64_t>(1, link_base[nf])), h_lvl(lvl_base[nf]);
  // tiles: 32 forests of similar step count per warp; all streams of a tile padded to its longest forest
  std::vector<uint32_t> tile_of(nf, 0);  // tile * 32 + lane
  std::vector<TileDesc> tiles;
  std::vector<uint32_t> h_ops_in, h_ops_out;
  {
    std::vector<uint32_t> tl;
    for (uint64_t i = 0; i < nf; ++i)
      if (in_tile[i]) tl.push_back((uint32_t)i);
    auto steps_in = [&](uint32_t i) { return ff[i].n_links + ff[i].n_real; };  // one header per node + one word per link
    std::stable_sort(tl.begin(), tl.end(), [&](uint32_t a, uint32_t x) { return steps_in(a) > steps_in(x); });
    tiles.resize((tl.size() + 31) / 32);
    uint64_t in_base = 0, out_base = 0, row_base = 0;
    for (size_t t = 0; t < tiles.size(); ++t) {
      TileDesc& T = tiles[t];
      std::memset(&T, 0, sizeof(T));
      uint64_t si = 0, so = 0, rows = 0;
      for (int l = 0; l < 32; ++l) {
        T.forest[l] = 0xffffffffu;
        const size_t k = t * 32 + l;
        if (k >= tl.size()) continue;
        const uint32_t i = tl[k];
        tile_of[i] = (uint32_t)k;
        si = std::max<uint64_t>(si, steps_in(i));
        so = std::max<uint64_t>(so, steps_in(i));
        rows = std::max<uint64_t>(rows, ff[i].n_real);
        bt->t_steps += 2 * (uint64_t)steps_in(i);
      }
      si = (si + 2 * kTileU - 1) / (2 * kTileU) * (2 * kTileU);
      so = (so + kTileU - 1) / kTileU * kTileU;
      T.ops_in_base = in_base;
      T.ops_out_base = out_base;
      T.row_base = row_base;
      T.steps_in = (uint32_t)si;
      T.steps_out = (uint32_t)so;
      in_base += si * 32;
      out_base += so * 32;
      row_base += rows * 32;
    }
    bt->n_tiles = (uint32_t)tiles.size();
    bt->t_forests = tl.size();
    bt->t_rows = row_base;
    h_ops_in.assign(in_base + (size_t)kTileAhead * kTileU * 32, kOpNop);  // + the prefetch tail
    h_ops_out.assign(out_base + (size_t)kTileAhead * kTileU * 32, kOpNop);
  }
  const bool no_stack = getenv("CML_FOREST_NO_STACK") != nullptr;  // tests / profiling: every value from global memory
  std::atomic<uint32_t> tile_stack_rows(2);  // shared-memory rows per lane the tile kernel needs (value / path stacks)
  std::vector<std::vector<uint64_t>> occ_parts(nt);
  {
    std::atomic<uint64_t> nextf(0);
    auto work = [&](unsigned tid) {
      ForestScratch S;
      std::vector<uint64_t>& occ = occ_parts[tid];
      occ.assign(f->rulespace, 0);
      for (;;) {
        const uint64_t i0 = nextf.fetch_add(64);
        if (i0 >= nf) break;
        for (uint64_t fi = i0; fi < std::min(nf, i0 + 64); ++fi) {
          const uint64_t o = b->node_off[fi];
          const uint32_t n = (uint32_t)(b->node_off[fi + 1] - o);
          const uint32_t* next = b->next + o;
          const uint32_t* label = b->label + o;
          const uint8_t* backref = b->backref + o;
          if (in_level[fi]) continue;  // (level tiles are laid out tile by tile below)
          FlatForest fx;
          forest_pass1(n, next, label, backref, f->rulespace, S, fx);  // recompute heights (cheap, keeps pass 1 memory small)
          const uint32_t nr = fx.n_real, nl = fx.n_levels;
          if (in_tile[fi]) {  // thread-per-forest tile: post-order numbering, transposed step streams
            const uint32_t t = tile_of[fi] >> 5, l = tile_of[fi] & 31;
            TileDesc& T = tiles[t];
            T.n_nodes[l] = nr;
            T.rows_out[l] = fx.n_links + nr;
            T.forest[l] = (uint32_t)fi;
            S.newid.assign(n, 0);
            for (uint32_t j = 0; j < nr; ++j) S.newid[S.post[j]] = j;
            uint32_t* oi = h_ops_in.data() + T.ops_in_base + l;
            uint32_t* oo = h_ops_out.data() + T.ops_out_base + l;
            // tree parent (the node a child is DEFINED in) and depth along tree parents; pre-order: parents first
            S.tpar.assign(n, 0xffffffffu);
            S.depth.assign(n, 0);
            uint32_t max_depth = 0;
            for (uint32_t p = 0; p < n; ++p) {
              if (backref[p]) continue;
              if (S.tpar[p] != 0xffffffffu) S.depth[p] = S.depth[S.tpar[p]] + 1;
              max_depth = std::max(max_depth, S.depth[p]);
              for (uint32_t q = p + 1; q < next[p]; q = next[q])
                if (!backref[q]) S.tpar[q] = p;
            }
            // stack mode: the post-order must be a proper walk of the tree children (simulate the value stack)
            bool stack_ok = max_depth <= (uint32_t)kDepthCap && !no_stack;
            uint32_t max_sp = 0;
            if (stack_ok) {
              S.sim.clear();
              for (uint32_t j = 0; j < nr && stack_ok; ++j) {
                const uint32_t p = S.post[j];
                S.kids.clear();
                for (uint32_t q = p + 1; q < next[p]; q = next[q])
                  if (!backref[q]) S.kids.push_back(q);
                for (size_t k = S.kids.size(); k-- > 0 && stack_ok;) {
                  if (S.sim.empty() || S.sim.back() != S.kids[k])
                    stack_ok = false;
                  else
                    S.sim.pop_back();
                }
                S.sim.push_back(p);
                max_sp = std::max<uint32_t>(max_sp, (uint32_t)S.sim.size());
              }
              if (max_sp > (uint32_t)kStackCap) stack_ok = false;
            }
            if (stack_ok) {
              uint32_t need = std::max(max_sp, 2 * (max_depth + 1));
              need += need & 1;
              uint32_t cur = tile_stack_rows.load();
              while (cur < need && !tile_stack_rows.compare_exchange_weak(cur, need)) {
              }
            }
            // parents per node: the inside header carries the count (7 bits) so the inside pass knows where the
            // node's header sits in the OUTSIDE stream (it leaves inside[node] there for the outside pass's prefetch)
            S.npar.assign(nr, 0);
            uint32_t max_par = 0;
            for (uint32_t j = 0; j < nr; ++j) {
              const uint32_t p = S.post[j];
              for (uint32_t q = p + 1; q < next[p]; q = next[q]) max_par = std::max(max_par, ++S.npar[S.newid[backref[q] ? label[q] : q]]);
            }
            const bool use_vout = max_par <= 127;
            if (!use_vout) T.rows_out[l] |= 0x80000000u;
            S.cnt.assign(nr + 1, 0);  // parent in-degrees -> offsets
            uint32_t s = 0;
            for (uint32_t j = 0; j < nr; ++j) {
              const uint32_t p = S.post[j];
              if (label[p]) ++occ[label[p]];
              const bool leaf = next[p] == p + 1;
              oi[(size_t)s++ * 32] = kHdr | (leaf ? kOpLast : 0u) | (stack_ok ? kHdrPush : 0u) |
                                     ((use_vout ? S.npar[j] : 0u) << kHdrNparShift) | label[p];
              if (leaf) continue;
              // links: children behind back references first (global reads), then the tree children, last defined
              // first (they are popped off the value stack)
              S.kids.clear();
              uint32_t n_links = 0;
              for (uint32_t q = p + 1; q < next[p]; q = next[q]) {
                ++n_links;
                ++S.cnt[S.newid[backref[q] ? label[q] : q] + 1];
                if (!backref[q] && stack_ok) S.kids.push_back(q);
              }
              uint32_t done = 0;
              for (uint32_t q = p + 1; q < next[p]; q = next[q]) {
                if (!backref[q] && stack_ok) continue;
                const uint32_t c = S.newid[backref[q] ? label[q] : q];
                oi[(size_t)s++ * 32] = c | (++done == n_links ? kOpLast : 0u);
              }
              for (size_t k = S.kids.size(); k-- > 0;)
                oi[(size_t)s++ * 32] = kLinkPop | (++done == n_links ? kOpLast : 0u);
            }
            for (uint32_t j = 0; j < nr; ++j) S.cnt[j + 1] += S.cnt[j];
            S.order.assign(S.cnt[nr] ? S.cnt[nr] : 1, 0);
            S.it.assign(nr, 0);
            for (uint32_t j = 0; j < nr; ++j) {  // parents in increasing post-order position => deterministic sums
              const uint32_t p = S.post[j];
              const uint32_t flag = label[p] ? 0u : kLinkOr;
              for (uint32_t q = p + 1; q < next[p]; q = next[q]) {
                const uint32_t c = S.newid[backref[q] ? label[q] : q];
                const uint32_t tree = (!backref[q] && stack_ok) ? kLinkTree : 0u;
                S.order[S.cnt[c] + S.it[c]++] = j | flag | tree;
              }
            }
            s = 0;
            for (uint32_t j = nr; j-- > 0;) {
              const uint32_t p = S.post[j];
              const uint32_t k0 = S.cnt[j], k1 = S.cnt[j + 1];
              const bool internal = next[p] != p + 1;
              oo[(size_t)s++ * 32] = kHdr | (k0 == k1 ? kOpLast : 0u) | (internal ? kHdrPush : 0u) |
                                     ((stack_ok ? S.depth[p] : 0u) << kHdrDepthShift) | label[p];
              for (uint32_t k = k0; k < k1; ++k) oo[(size_t)s++ * 32] = S.order[k] | (k + 1 == k1 ? kOpLast : 0u);
            }
            continue;
          }
          // counting sort by height, stable in pre-order
          S.cnt.assign(nl + 1, 0);
          for (uint32_t i = 0; i < n; ++i)
            if (!backref[i]) ++S.cnt[S.height[i] + 1];
          for (uint32_t L = 0; L < nl; ++L) S.cnt[L + 1] += S.cnt[L];
          uint32_t* lvl = h_lvl.data() + lvl_base[fi];
          for (uint32_t L = 0; L <= nl; ++L) lvl[L] = S.cnt[L];
          S.newid.assign(n, 0);
          S.order.assign(nr, 0);
          for (uint32_t i = 0; i < n; ++i)
            if (!backref[i]) {
              const uint32_t id = S.cnt[S.height[i]]++;
              S.newid[i] = id;
              S.order[id] = i;
            }
          uint32_t* lab = h_label.data() + node_base[fi];
          uint32_t* coff = h_coff.data() + node_base[fi];
          uint32_t* poff = h_poff.data() + node_base[fi];
          uint32_t* child = h_child.data() + link_base[fi];
          uint32_t* par = h_par.data() + link_base[fi];
          // children CSR in the new order; parent in-degrees
          std::fill(poff, poff + nr + 1, 0u);
          uint32_t nc = 0;
          for (uint32_t id = 0; id < nr; ++id) {
            const uint32_t p = S.order[id];
            lab[id] = label[p];
            if (label[p]) ++occ[label[p]];
            coff[id] = nc;
            for (uint32_t q = p + 1; q < next[p]; q = next[q]) {
              const uint32_t c = S.newid[backref[q] ? label[q] : q];
              child[nc++] = c;
              ++poff[c + 1];
            }
          }
          coff[nr] = nc;
          lab[nr] = 0;
          for (uint32_t id = 0; id < nr; ++id) poff[id + 1] += poff[id];
          S.it.assign(nr, 0);
          for (uint32_t id = 0; id < nr; ++id) {  // parents in increasing internal order => deterministic sums
            const uint32_t flag = lab[id] ? 0u : kHotBit;
            for (uint32_t k = coff[id]; k < coff[id + 1]; ++k) {
              const uint32_t c = child[k];
              par[poff[c] + S.it[c]++] = id | flag;
            }
          }
          ForestDesc& d = desc[fi];
          d.node_base = node_base[fi];
          d.child_base = d.par_base = link_base[fi];
          d.lvl_base = lvl_base[fi];
          d.n_nodes = nr;
          d.n_levels = nl;
          d.index = (uint32_t)fi;
          d.pad = 0;
        }
      }
    };
    std::vector<std::thread> th;
    for (unsigned t = 1; t < nt; ++t) th.emplace_back(work, t);
    work(0);
    for (auto& t : th) t.join();
  }
  // ---- level tiles: per tile, the nodes of its forests height-major (level, forest, pre-order), two CSRs of 16-bit local ids
  const size_t n_lt = lv_first.empty() ? 0 : lv_first.size() - 1;
  std::vector<LevelTile> ltiles(n_lt);
  std::vector<uint32_t> lt_label, lt_coff, lt_poff, lt_lvl, lt_forest(lv_forests.size());
  std::vector<uint16_t> lt_child, lt_par, lt_root(lv_forests.size());
  if (n_lt) {
    uint64_t nb = 0, lb = 0, vb = 0;
    for (size_t t = 0; t < n_lt; ++t) {
      LevelTile& T = ltiles[t];
      std::memset(&T, 0, sizeof(T));
      T.node_base = nb;
      T.link_base = lb;
      T.lvl_base = vb;
      T.forest_base = lv_first[t];
      T.n_forests = lv_first[t + 1] - lv_first[t];
      uint32_t nn = 0, nlv = 0;
      uint64_t nk = 0;
      for (uint32_t k = lv_first[t]; k < lv_first[t + 1]; ++k) {
        const uint32_t fi = lv_forests[k];
        nn += ff[fi].n_real;
        nk += ff[fi].n_links;
        nlv = std::max(nlv, ff[fi].n_levels);
      }
      T.n_nodes = nn;
      T.n_levels = nlv;
      nb += nn + 1;
      lb += nk;
      vb += 3ull * (nlv + 1);
      if (t < lv_n_small)
        bt->lt_small_nodes = std::max(bt->lt_small_nodes, nn);
      else
        bt->lt_max_nodes = std::max(bt->lt_max_nodes, nn);
      bt->lt_max_levels = std::max(bt->lt_max_levels, nlv);
      bt->lt_nodes += nn;
      bt->lt_links += nk;
    }
    bt->n_ltiles = (uint32_t)n_lt;
    bt->n_stiles = lv_n_small;
    bt->lt_forests = lv_forests.size();
    lt_label.assign(nb + 16, 0);
    lt_coff.assign(nb + 16, 0);
    lt_poff.assign(nb + 16, 0);
    lt_lvl.assign(vb, 0);
    lt_child.assign(lb + 16, 0);
    lt_par.assign(lb + 16, 0);
    std::atomic<size_t> next_tile(0);
    std::atomic<int> tile_err(0);
    auto work = [&](unsigned tid) {
      ForestScratch S;
      std::vector<uint64_t>& occ = occ_parts[tid];
      if (occ.size() != f->rulespace) occ.assign(f->rulespace, 0);
      std::vector<uint32_t> H, newid, cnt, pre_off, itp;
      for (;;) {
        const size_t t = next_tile.fetch_add(1);
        if (t >= n_lt) break;
        const LevelTile& T = ltiles[t];
        const uint32_t nft = T.n_forests, nlv = T.n_levels, nn = T.n_nodes;
        uint32_t* lab = lt_label.data() + T.node_base;
        uint32_t* coff = lt_coff.data() + T.node_base;
        uint32_t* poff = lt_poff.data() + T.node_base;
        uint16_t* child = lt_child.data() + T.link_base;
        uint16_t* par = lt_par.data() + T.link_base;
        uint32_t* lvl = lt_lvl.data() + T.lvl_base;
        cnt.assign((size_t)nlv * nft, 0);
        H.clear();
        pre_off.assign(nft + 1, 0);
        for (uint32_t k = 0; k < nft; ++k) {  // heights of every pre-order node of the tile; nodes per (level, forest)
          const uint32_t fi = lv_forests[T.forest_base + k];
          const uint64_t o = b->node_off[fi];
          const uint32_t n = (uint32_t)(b->node_off[fi + 1] - o);
          FlatForest fx;
          forest_pass1(n, b->next + o, b->label + o, b->backref + o, f->rulespace, S, fx);
          if (fx.error) tile_err = 1;
          pre_off[k + 1] = pre_off[k] + n;
          H.insert(H.end(), S.height.begin(), S.height.begin() + n);
          const uint8_t* backref = b->backref + o;
          for (uint32_t i = 0; i < n; ++i)
            if (!backref[i]) ++cnt[(size_t)S.height[i] * nft + k];
        }
        uint32_t run = 0;
        for (uint32_t L = 0; L < nlv; ++L) {
          lvl[L] = run;
          for (uint32_t k = 0; k < nft; ++k) {
            const uint32_t c = cnt[(size_t)L * nft + k];
            cnt[(size_t)L * nft + k] = run;
            run += c;
          }
        }
        lvl[nlv] = run;
        newid.assign(pre_off[nft], 0);
        std::fill(coff, coff + nn + 1, 0u);
        std::fill(poff, poff + nn + 1, 0u);
        for (uint32_t k = 0; k < nft; ++k) {  // local ids, stable in pre-order within (level, forest)
          const uint32_t fi = lv_forests[T.forest_base + k];
          const uint64_t o = b->node_off[fi];
          const uint32_t n = pre_off[k + 1] - pre_off[k];
          const uint8_t* backref = b->backref + o;
          for (uint32_t i = 0; i < n; ++i)
            if (!backref[i]) newid[pre_off[k] + i] = cnt[(size_t)H[pre_off[k] + i] * nft + k]++;
          lt_root[T.forest_base + k] = (uint16_t)newid[pre_off[k]];
          lt_forest[T.forest_base + k] = fi;
        }
        for (uint32_t k = 0; k < nft; ++k) {  // labels, child / parent degrees
          const uint32_t fi = lv_forests[T.forest_base + k];
          const uint64_t o = b->node_off[fi];
          const uint32_t n = pre_off[k + 1] - pre_off[k];
          const uint32_t* next = b->next + o;
          const uint32_t* label = b->label + o;
          const uint8_t* backref = b->backref + o;
          const uint32_t* nid = newid.data() + pre_off[k];
          for (uint32_t p = 0; p < n; ++p) {
            if (backref[p]) continue;
            const uint32_t id = nid[p];
            lab[id] = label[p];
            if (label[p]) ++occ[label[p]];
            for (uint32_t q = p + 1; q < next[p]; q = next[q]) {
              ++coff[id + 1];
              ++poff[nid[backref[q] ? label[q] : q] + 1];
            }
          }
        }
        for (uint32_t id = 0; id < nn; ++id) {
          coff[id + 1] += coff[id];
          poff[id + 1] += poff[id];
        }
        for (uint32_t L = 0; L <= nlv; ++L) {
          lvl[(nlv + 1) + L] = coff[lvl[L]];
          lvl[2 * (nlv + 1) + L] = poff[lvl[L]];
        }
        itp.assign(nn, 0);
        for (uint32_t k = 0; k < nft; ++k) {  // links: children in the reference's order; parents in (forest, pre-order) order
          const uint32_t fi = lv_forests[T.forest_base + k];
          const uint64_t o = b->node_off[fi];
          const uint32_t n = pre_off[k + 1] - pre_off[k];
          const uint32_t* next = b->next + o;
          const uint32_t* label = b->label + o;
          const uint8_t* backref = b->backref + o;
          const uint32_t* nid = newid.data() + pre_off[k];
          for (uint32_t p = 0; p < n; ++p) {
            if (backref[p]) continue;
            const uint32_t id = nid[p];
            const uint32_t flag = label[p] ? 0u : kLvlOrParent;
            uint32_t kk = coff[id];
            for (uint32_t q = p + 1; q < next[p]; q = next[q]) {
              const uint32_t c = nid[backref[q] ? label[q] : q];
              child[kk++] = (uint16_t)c;
              par[poff[c] + itp[c]++] = (uint16_t)(id | flag);
            }
          }
        }
      }
    };
    std::vector<std::thread> th;
    for (unsigned t = 1; t < nt; ++t) th.emplace_back(work, t);
    work(0);
    for (auto& t : th) t.join();
    F_REQUIRE(!tile_err.load(), CML_ERR_ARG, "cml_forests_add: forest changed between passes");
  }
  for (auto const& occ : occ_parts)
    for (uint64_t r = 0; r < occ.size(); ++r) f->rule_occ[r] += occ[r];
  // classes: smallest shared-memory capacity that fits, else the CTA class
  const size_t real_b = f->precision == 64 ? 8 : 4;
  std::vector<std::vector<uint32_t>> by_cls(kNWarpCls + 1);
  for (uint64_t i = 0; i < nf; ++i) {
    if (in_tile[i] || in_level[i]) continue;
    int c = kNWarpCls;
    for (int k = 0; k < kNWarpCls; ++k)
      if (desc[i].n_nodes <= kWarpCaps[k] && (size_t)kWarpsPerCta * 2 * kWarpCaps[k] * real_b <= f->smem_optin) {
        c = k;
        break;
      }
    by_cls[c].push_back((uint32_t)i);
  }
  std::vector<uint32_t> list;
  for (int c = 0; c <= kNWarpCls; ++c) {
    bt->cls_begin[c] = (uint32_t)list.size();
    // largest first: the tail of a class is then made of short forests
    std::stable_sort(by_cls[c].begin(), by_cls[c].end(), [&](uint32_t a, uint32_t x) { return desc[a].n_nodes > desc[x].n_nodes; });
    list.insert(list.end(), by_cls[c].begin(), by_cls[c].end());
  }
  bt->cls_begin[kNWarpCls + 1] = (uint32_t)list.size();
  const uint32_t n_cta = bt->cls_begin[kNWarpCls + 1] - bt->cls_begin[kNWarpCls];
  if (n_cta) {
    bt->scratch_stride = (bt->max_nodes + 31) & ~31ull;
    bt->cta_grid = std::min<uint32_t>(n_cta, 2 * f->sm_count);
    CML_CUDA(bt->scratch.alloc((size_t)bt->cta_grid * 2 * bt->scratch_stride * real_b));
  }
  CML_CUDA(bt->desc.upload(desc.data(), desc.size(), f->stream));
  CML_CUDA(bt->label.upload(h_label.data(), h_label.size(), f->stream));
  CML_CUDA(bt->child_off.upload(h_coff.data(), h_coff.size(), f->stream));
  CML_CUDA(bt->par_off.upload(h_poff.data(), h_poff.size(), f->stream));
  CML_CUDA(bt->child.upload(h_child.data(), link_base[nf], f->stream));
  CML_CUDA(bt->par.upload(h_par.data(), link_base[nf], f->stream));
  CML_CUDA(bt->lvl_off.upload(h_lvl.data(), h_lvl.size(), f->stream));
  CML_CUDA(bt->list.upload(list.data(), list.size(), f->stream));
  if (bt->n_tiles) {
    CML_CUDA(bt->tiles.upload(tiles.data(), tiles.size(), f->stream));
    CML_CUDA(bt->t_ops_in.upload(h_ops_in.data(), h_ops_in.size(), f->stream));
    CML_CUDA(bt->t_ops_out.upload(h_ops_out.data(), h_ops_out.size(), f->stream));
    bt->t_stack_rows = tile_stack_rows.load();
    CML_CUDA(bt->t_in.alloc(bt->t_rows * real_b));
    CML_CUDA(bt->t_ga.alloc(bt->t_rows * real_b));
    CML_CUDA(bt->t_vout.alloc(h_ops_out.size() * real_b));  // one value slot per outside stream word
    CML_CUDA(cudaMemsetAsync(bt->t_vout.p, 0, h_ops_out.size() * real_b, f->stream));
  }
  if (bt->n_ltiles) {
    CML_CUDA(bt->ltiles.upload(ltiles.data(), ltiles.size(), f->stream));
    CML_CUDA(bt->lt_label.upload(lt_label.data(), lt_label.size(), f->stream));
    CML_CUDA(bt->lt_coff.upload(lt_coff.data(), lt_coff.size(), f->stream));
    CML_CUDA(bt->lt_poff.upload(lt_poff.data(), lt_poff.size(), f->stream));
    CML_CUDA(bt->lt_lvl.upload(lt_lvl.data(), lt_lvl.size(), f->stream));
    CML_CUDA(bt->lt_child.upload(lt_child.data(), lt_child.size(), f->stream));
    CML_CUDA(bt->lt_par.upload(lt_par.data(), lt_par.size(), f->stream));
    CML_CUDA(bt->lt_root.upload(lt_root.data(), lt_root.size(), f->stream));
    CML_CUDA(bt->lt_forest.upload(lt_forest.data(), lt_forest.size(), f->stream));
  }
  CML_CUDA(bt->ln_inside.alloc(nf));
  CML_CUDA(cudaEventCreate(&bt->ev0));
  CML_CUDA(cudaEventCreate(&bt->ev1));
  CML_CUDA(cudaStreamSynchronize(f->stream));
  f->batches.push_back(std::move(bt));
  f->hot_dirty = true;
  return CML_OK;
}

extern "C" int cml_forests_totals(cml_forests* f, uint64_t* n_forests, uint64_t* n_nodes, uint64_t* n_hyperedges, uint64_t* n_links) {
  if (!f) return CML_ERR_ARG;
  uint64_t a = 0, b = 0, c = 0, d = 0;
  for (auto const& bt : f->batches) {
    a += bt->n_forests;
    b += bt->n_nodes;
    c += bt->n_hyperedges;
    d += bt->n_links;
  }
  if (n_forests) *n_forests = a;
  if (n_nodes) *n_nodes = b;
  if (n_hyperedges) *n_hyperedges = c;
  if (n_links) *n_links = d;
  return CML_OK;
}

static int forest_rebuild_hot(cml_forests* f) {
  uint64_t min_occ = 4096;
  uint32_t max_hot = 8192;
  if (const char* e = getenv("CML_FOREST_HOT_MIN_OCC")) min_occ = std::strtoull(e, nullptr, 10);
  if (const char* e = getenv("CML_FOREST_HOT_MAX")) max_hot = (uint32_t)std::strtoul(e, nullptr, 10);
  std::vector<uint32_t> hot_rule;
  for (uint64_t r = 1; r < f->rulespace; ++r)
    if (f->rule_occ[r] >= min_occ) hot_rule.push_back((uint32_t)r);
  if (hot_rule.size() > max_hot) {
    std::partial_sort(hot_rule.begin(), hot_rule.begin() + max_hot, hot_rule.end(),
                      [&](uint32_t a, uint32_t b) { return f->rule_occ[a] > f->rule_occ[b] || (f->rule_occ[a] == f->rule_occ[b] && a < b); });
    hot_rule.resize(max_hot);
  }
  std::vector<uint32_t> hot_index(f->rulespace, 0xFFFFFFFFu);
  for (size_t h = 0; h < hot_rule.size(); ++h) hot_index[hot_rule[h]] = (uint32_t)h;
  f->n_hot = (uint32_t)hot_rule.size();
  CML_CUDA(f->hot_index.upload(hot_index.data(), hot_index.size(), f->stream));
  CML_CUDA(f->hot_rule.upload(hot_rule.data(), hot_rule.size(), f->stream));
  CML_CUDA(f->hot.alloc(std::max<size_t>(1, (size_t)kHotCopies * f->n_hot)));
  for (auto& bt : f->batches) {
    if (bt->n_forests > bt->t_forests + bt->lt_forests) {  // (only batches that hold per-forest CSRs)
      k_forest_mark_hot<<<f_cdiv(bt->label.n, 256), 256, 0, f->stream>>>(bt->label.n, bt->label.p, f->hot_index.p);
      ++f->launches;
    }
    if (bt->n_ltiles) {
      if (!bt->lt_label_out.p) CML_CUDA(bt->lt_label_out.alloc(bt->lt_label.n));
      k_forest_label_out<<<f_cdiv(bt->lt_label.n, 256), 256, 0, f->stream>>>(bt->lt_label.n, bt->lt_label.p, f->hot_index.p,
                                                                          bt->lt_label_out.p);
      ++f->launches;
    }
    if (bt->n_tiles) {
      k_forest_mark_hot_ops<<<f_cdiv(bt->t_ops_out.n, 256), 256, 0, f->stream>>>(bt->t_ops_out.n, bt->t_ops_out.p,
                                                                               f->hot_index.p);
      ++f->launches;
    }
  }
  CML_CUDA(cudaGetLastError());
  CML_CUDA(cudaStreamSynchronize(f->stream));
  f->hot_dirty = false;
  return CML_OK;
}

template <typename Real>
static int forest_launch(cml_forests* f, ForestBatch& bt) {
  ForestArgs A{};
  A.desc = bt.desc.p;
  A.label = bt.label.p;
  A.child_off = bt.child_off.p;
  A.par_off = bt.par_off.p;
  A.child = bt.child.p;
  A.par = bt.par.p;
  A.lvl_off = bt.lvl_off.p;
  A.lnw = f->w_real.p;
  A.hot_index = f->hot_index.p;
  A.counts = f->reduce.p;
  A.hot = f->hot.p;
  A.n_hot = f->n_hot;
  A.ln_inside = bt.ln_inside.p;
  bt.n_kernels = 0;
  CML_CUDA(cudaEventRecord(bt.ev0, f->stream));
  if (bt.n_tiles) {
    TileArgs T{};
    T.tiles = bt.tiles.p;
    T.n_tiles = bt.n_tiles;
    T.ops_in = bt.t_ops_in.p;
    T.ops_out = bt.t_ops_out.p;
    T.in_ = bt.t_in.p;
    T.ga = bt.t_ga.p;
    T.lnw = f->w_real.p;
    T.hot_index = f->hot_index.p;
    T.counts = f->reduce.p;
    T.hot = f->hot.p;
    T.n_hot = f->n_hot;
    T.ln_inside = bt.ln_inside.p;
    T.stack_rows = bt.t_stack_rows;
    const size_t tsmem = (size_t)kTileWarps * bt.t_stack_rows * 32 * sizeof(Real) +
                         (size_t)kTileWarps * kTileStages * kTileU * 32 * (sizeof(uint32_t) + sizeof(Real));
    T.vout = bt.t_vout.p;
    if (tsmem > 48 * 1024)
      CML_CUDA(cudaFuncSetAttribute(k_forest_thread<Real>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tsmem));
    k_forest_thread<Real><<<f_cdiv(bt.n_tiles, kTileWarps), kTileWarps * 32, tsmem, f->stream>>>(T);
    ++f->launches;
    ++bt.n_kernels;
  }
  if (bt.n_ltiles) {
    LevelArgs L{};
    L.tiles = bt.ltiles.p;
    L.label = bt.lt_label.p;
    L.label_out = bt.lt_label_out.p;
    L.coff = bt.lt_coff.p;
    L.poff = bt.lt_poff.p;
    L.child = bt.lt_child.p;
    L.par = bt.lt_par.p;
    L.lvl = bt.lt_lvl.p;
    L.root = bt.lt_root.p;
    L.forest = bt.lt_forest.p;
    L.lnw = f->w_real.p;
    L.hot_index = f->hot_index.p;
    L.counts = f->reduce.p;
    L.hot = f->hot.p;
    L.n_hot = f->n_hot;
    L.ln_inside = bt.ln_inside.p;
    L.pf = 2;
    if (const char* e = getenv("CML_FOREST_LEVEL_PREFETCH")) L.pf = std::max(0, atoi(e));
    // launch shapes (threads x resident CTAs per SM, nodes in flight per thread).  Small tiles: 128 x 16 x 1 by default
    // (CML_FOREST_LEVEL_VARIANT picks another shape for measurements; the tile capacity CML_FOREST_LEVEL_SMEM_KB at add
    // time decides how many CTAs really fit); large tiles: 512 x 2 x 4.
    int variant = 6;
    if (const char* e = getenv("CML_FOREST_LEVEL_VARIANT")) variant = atoi(e);
    auto go = [&](auto kern, int threads, uint32_t first, uint32_t n, uint32_t max_nodes) -> int {
      const size_t vsmem = ((size_t)max_nodes * sizeof(Real) + 15) & ~(size_t)15;
      const size_t lsmem = vsmem + ((12 * ((size_t)bt.lt_max_levels + 1) + 15) & ~(size_t)15);
      LevelArgs X = L;
      X.tiles = bt.ltiles.p + first;
      X.n_tiles = n;
      X.cap = max_nodes;
      X.lvl_smem_off = (uint32_t)vsmem;
      CML_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)std::max<size_t>(lsmem, 48 * 1024)));
      kern<<<n, threads, lsmem, f->stream>>>(X);
      ++f->launches;
      ++bt.n_kernels;
      return CML_OK;
    };
    if (bt.n_stiles) {
      const uint32_t n = bt.n_stiles, mx = bt.lt_small_nodes;
      int rc;
      switch (variant) {
        case 0: rc = go(k_forest_level<Real, 512, 2, 4>, 512, 0, n, mx); break;
        case 1: rc = go(k_forest_level<Real, 384, 3, 4>, 384, 0, n, mx); break;
        case 2: rc = go(k_forest_level<Real, 256, 4, 4>, 256, 0, n, mx); break;
        case 3: rc = go(k_forest_level<Real, 256, 6, 2>, 256, 0, n, mx); break;
        case 4: rc = go(k_forest_level<Real, 128, 12, 2>, 128, 0, n, mx); break;
        case 5: rc = go(k_forest_level<Real, 256, 8, 1>, 256, 0, n, mx); break;
        case 7: rc = go(k_forest_level<Real, 64, 24, 2>, 64, 0, n, mx); break;
        default: rc = go(k_forest_level<Real, 128, 16, 1>, 128, 0, n, mx);
      }
      if (rc) return rc;
    }
    if (bt.n_ltiles > bt.n_stiles) {
      const int rc = go(k_forest_level<Real, 512, 2, 4>, 512, bt.n_stiles, bt.n_ltiles - bt.n_stiles, bt.lt_max_nodes);
      if (rc) return rc;
    }
  }
  for (int c = 0; c < kNWarpCls; ++c) {
    const uint32_t n = bt.cls_begin[c + 1] - bt.cls_begin[c];
    if (!n) continue;
    A.list = bt.list.p + bt.cls_begin[c];
    A.n_list = n;
    A.cap = kWarpCaps[c];
    const size_t smem = (size_t)kWarpsPerCta * 2 * A.cap * sizeof(Real);
    if (smem > 48 * 1024) CML_CUDA(cudaFuncSetAttribute(k_forest_warp<Real>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    // a few forests per warp so the short tail of the (size-sorted) class balances the long head
    const unsigned grid = std::max(1u, std::min(f_cdiv(n, kWarpsPerCta), (unsigned)f->sm_count * 16u));
    k_forest_warp<Real><<<grid, kWarpsPerCta * 32, smem, f->stream>>>(A);
    ++f->launches;
    ++bt.n_kernels;
  }
  {
    const uint32_t n = bt.cls_begin[kNWarpCls + 1] - bt.cls_begin[kNWarpCls];
    if (n) {
      A.list = bt.list.p + bt.cls_begin[kNWarpCls];
      A.n_list = n;
      A.scratch = bt.scratch.p;
      A.scratch_stride = bt.scratch_stride;
      k_forest_cta<Real><<<bt.cta_grid, kCtaThreads, 0, f->stream>>>(A);
      ++f->launches;
      ++bt.n_kernels;
    }
  }
  CML_CUDA(cudaEventRecord(bt.ev1, f->stream));
  CML_CUDA(cudaGetLastError());
  return CML_OK;
}

extern "C" int cml_forests_estimate_launch(cml_forests* f) {
  if (!f) return CML_ERR_ARG;
  F_REQUIRE(f->have_params, CML_ERR_STATE, "cml_forests_estimate before cml_forests_set_params");
  CML_CUDA(cudaSetDevice(f->device));
  if (f->hot_dirty) {
    const int rc = forest_rebuild_hot(f);
    if (rc) return rc;
  }
  if (f->precision == 64)
    k_forest_cast_w<double><<<f_cdiv(f->rulespace, 256), 256, 0, f->stream>>>(f->rulespace, f->ln_w.p, (double*)f->w_real.p);
  else
    k_forest_cast_w<float><<<f_cdiv(f->rulespace, 256), 256, 0, f->stream>>>(f->rulespace, f->ln_w.p, (float*)f->w_real.p);
  ++f->launches;
  CML_CUDA(cudaMemsetAsync(f->reduce.p, 0, (f->rulespace + 3) * sizeof(double), f->stream));
  if (f->n_hot) CML_CUDA(cudaMemsetAsync(f->hot.p, 0, (size_t)kHotCopies * f->n_hot * sizeof(double), f->stream));
  for (auto& bt : f->batches) {
    const int rc = f->precision == 64 ? forest_launch<double>(f, *bt) : forest_launch<float>(f, *bt);
    if (rc) return rc;
    if (!f->sum_partial.p) CML_CUDA(f->sum_partial.alloc(2 * kSumBlocks));
    k_forest_sum_partial<<<kSumBlocks, 256, 0, f->stream>>>(bt->ln_inside.p, bt->n_forests, f->sum_partial.p);
    k_forest_sum<<<1, 256, 0, f->stream>>>(f->sum_partial.p, kSumBlocks, f->reduce.p + f->rulespace, bt->n_forests);
    f->launches += 2;
  }
  if (f->n_hot) {
    k_forest_fold<<<f_cdiv(f->n_hot, 128), 128, 0, f->stream>>>(f->n_hot, f->hot_rule.p, f->hot.p, f->reduce.p);
    ++f->launches;
  }
  CML_CUDA(cudaGetLastError());
  f->pending = true;
  return CML_OK;
}
extern "C" int cml_forests_estimate_finish(cml_forests* f, cml_forest_estimate_result* out) {
  if (!f) return CML_ERR_ARG;
  F_REQUIRE(f->pending, CML_ERR_STATE, "cml_forests_estimate_finish without a launched estimate");
  CML_CUDA(cudaSetDevice(f->device));
  double scal[3];
  CML_CUDA(cudaMemcpyAsync(scal, f->reduce.p + f->rulespace, sizeof(scal), cudaMemcpyDeviceToHost, f->stream));
  CML_CUDA(cudaStreamSynchronize(f->stream));
  f->pending = false;
  if (out) {
    out->sum_ln_p = scal[0];
    out->n_zero = (uint64_t)(scal[1] + 0.5);
    out->n_forests = (uint64_t)(scal[2] + 0.5);
  }
  return CML_OK;
}
extern "C" int cml_forests_estimate(cml_forests* f, cml_forest_estimate_result* out) {
  const int rc = cml_forests_estimate_launch(f);
  if (rc) return rc;
  return cml_forests_estimate_finish(f, out);
}
extern "C" int cml_forests_last_time_ms(cml_forests* f, float* ms, uint32_t* n_kernels) {
  if (!f) return CML_ERR_ARG;
  float total = 0;
  uint32_t nk = 0;
  for (auto& bt : f->batches) {
    float t = 0;
    CML_CUDA(cudaEventSynchronize(bt->ev1));
    CML_CUDA(cudaEventElapsedTime(&t, bt->ev0, bt->ev1));
    total += t;
    nk += bt->n_kernels;
  }
  if (ms) *ms = total;
  if (n_kernels) *n_kernels = nk;
  return CML_OK;
}
extern "C" int cml_forests_get_inside(cml_forests* f, double* ln_inside, uint64_t n) {
  if (!f || !ln_inside) return CML_ERR_ARG;
  CML_CUDA(cudaSetDevice(f->device));
  uint64_t o = 0;
  for (auto& bt : f->batches) {
    F_REQUIRE(o + bt->n_forests <= n, CML_ERR_ARG, "cml_forests_get_inside: buffer too small");
    CML_CUDA(cudaMemcpyAsync(ln_inside + o, bt->ln_inside.p, bt->n_forests * sizeof(double), cudaMemcpyDeviceToHost, f->stream));
    o += bt->n_forests;
  }
  CML_CUDA(cudaStreamSynchronize(f->stream));
  return CML_OK;
}
// ---------------------------------------------------------------------------------------------------
// Viterbi (best derivation) over the forests in the reference's own representation: FForest::viterbi_rec
// (forest-em/forest.hpp:507-574): as inside, with max at the OR nodes; best[i] = the chosen child of OR node i (the
// first child that attains the maximum).  A decode-side pass that runs once after training (forest-em -v): one thread
// per forest, the recursion as an explicit stack of open nodes over the pre-order array.
// ---------------------------------------------------------------------------------------------------
const int kVitDepth = 96;
__global__ void k_forest_viterbi(uint64_t n_forests, const uint64_t* __restrict__ node_off, const uint32_t* __restrict__ next,
                                 const uint32_t* __restrict__ label, const uint8_t* __restrict__ backref,
                                 const double* __restrict__ ln_w, double* __restrict__ vit, uint32_t* __restrict__ best,
                                 double* __restrict__ root, int* __restrict__ err) {
  const uint64_t f = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (f >= n_forests) return;
  const uint64_t base = node_off[f];
  const uint32_t n = (uint32_t)(node_off[f + 1] - base);
  const uint32_t* nx = next + base;
  const uint32_t* lb = label + base;
  const uint8_t* br = backref + base;
  double* v = vit + base;
  uint32_t* bc = best + base;
  uint32_t s_node[kVitDepth];
  double s_acc[kVitDepth];
  uint32_t s_best[kVitDepth];
  int sp = 0;
  for (uint32_t i = 0; i < n; ++i) {
    double val;
    bool done;
    if (br[i]) {
      val = v[lb[i]];  // a shared sub-forest: defined (and finished) earlier in the pre-order
      v[i] = val;
      done = true;
    } else if (nx[i] == i + 1) {
      val = lb[i] ? ln_w[lb[i]] : -CUDART_INF;  // leaf rule (an OR node without children cannot be written)
      v[i] = val;
      done = true;
    } else {
      if (sp >= kVitDepth) {
        *err = 1;
        return;
      }
      s_node[sp] = i;
      s_acc[sp] = lb[i] ? ln_w[lb[i]] : -CUDART_INF;
      s_best[sp] = 0xFFFFFFFFu;
      ++sp;
      done = false;
      val = 0;
    }
    uint32_t child = i;
    while (done && sp > 0) {  // hand the finished value to the open parent; close parents that end here
      const int t = sp - 1;
      const uint32_t p = s_node[t];
      if (lb[p]) {
        s_acc[t] += val;
      } else if (s_best[t] == 0xFFFFFFFFu || val > s_acc[t]) {
        s_acc[t] = val;
        s_best[t] = child;
      }
      if (nx[p] == i + 1) {  // the parent's last descendant was node i
        val = s_acc[t];
        v[p] = val;
        bc[p] = s_best[t];
        child = p;
        --sp;
      } else
        done = false;
    }
  }
  root[f] = n ? v[0] : -CUDART_INF;
}

// viterbi scores (ln) of every forest's root and, per node of the batch, the chosen child of OR nodes (in-forest
// pre-order index; 0xFFFFFFFF elsewhere), at the current rule weights.  The batch is the one given to cml_forests_add
// (the device keeps forests in its own layouts, so the reference arrays are uploaded again for this one-off pass).
extern "C" int cml_forests_viterbi(cml_forests* f, const cml_forest_batch* b, double* root_ln, uint32_t* best_child) {
  if (!f || !b || !root_ln || !best_child) return CML_ERR_ARG;
  F_REQUIRE(f->have_params, CML_ERR_STATE, "cml_forests_viterbi before cml_forests_set_params");
  CML_CUDA(cudaSetDevice(f->device));
  if (!b->n_forests) return CML_OK;
  const uint64_t n_nodes = b->node_off[b->n_forests];
  DevArray<uint64_t> d_off;
  DevArray<uint32_t> d_next, d_label, d_best;
  DevArray<uint8_t> d_br;
  DevArray<double> d_vit, d_root;
  DevArray<int> d_err;
  cudaStream_t s = f->stream;
  CML_CUDA(d_off.upload(b->node_off, b->n_forests + 1, s));
  CML_CUDA(d_next.upload(b->next, n_nodes, s));
  CML_CUDA(d_label.upload(b->label, n_nodes, s));
  CML_CUDA(d_br.upload(b->backref, n_nodes, s));
  CML_CUDA(d_best.alloc(std::max<uint64_t>(1, n_nodes)));
  CML_CUDA(d_vit.alloc(std::max<uint64_t>(1, n_nodes)));
  CML_CUDA(d_root.alloc(b->n_forests));
  CML_CUDA(d_err.alloc(1));
  CML_CUDA(cudaMemsetAsync(d_err.p, 0, sizeof(int), s));
  CML_CUDA(cudaMemsetAsync(d_best.p, 0xFF, std::max<uint64_t>(1, n_nodes) * sizeof(uint32_t), s));
  k_forest_viterbi<<<f_cdiv(b->n_forests, 128), 128, 0, s>>>(b->n_forests, d_off.p, d_next.p, d_label.p, d_br.p, f->ln_w.p, d_vit.p,
                                                             d_best.p, d_root.p, d_err.p);
  ++f->launches;
  CML_CUDA(cudaGetLastError());
  int herr = 0;
  CML_CUDA(cudaMemcpyAsync(&herr, d_err.p, sizeof(int), cudaMemcpyDeviceToHost, s));
  CML_CUDA(cudaMemcpyAsync(root_ln, d_root.p, b->n_forests * sizeof(double), cudaMemcpyDeviceToHost, s));
  CML_CUDA(cudaMemcpyAsync(best_child, d_best.p, n_nodes * sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
  CML_CUDA(cudaStreamSynchronize(s));
  F_REQUIRE(!herr, CML_ERR_ARG, "cml_forests_viterbi: a forest nests deeper than 96 levels");
  return CML_OK;
}
// ---------------------------------------------------------------------------------------------------
// forest-em --crp: Gibbs sampling of one derivation per forest under the CRP cache model.
// Reference: FForests::resample_block (forest-em/forest-em.hpp:752-764): FForest::compute_inside(W) with the proposal
// probabilities count/normsum (forest.hpp:769-816), then FForest::choose_random top-down (forest.hpp:726-758): at an OR
// node one uniform picks the first child whose (inside^power / norm) takes the running choice below zero, an AND node
// records its rule and descends into all children; a back reference continues with power 1 (reproduced).  Counts:
// gibbs_base::iteration (graehl/shared/gibbs.hpp:836-877).  Uniforms are counter based, u(seed, sweep, forest, draw),
// one per OR node visited, in visit order, so SEQUENTIAL mode reproduces the CPU restatement derivation by derivation.
// The sampler works on the reference's pre-order arrays (the recursion as explicit stacks); arithmetic is the
// reference's fp64 logweight (pairwise log-add in child order).
// ---------------------------------------------------------------------------------------------------
const int kGibbsDepth = 96, kGibbsStack = 384;
__device__ __forceinline__ double fg_uniform(uint64_t seed, uint32_t sweep, uint32_t block, uint32_t draw) {
  uint64_t h = mix64(seed ^ mix64(((uint64_t)sweep << 32) | block));
  h = mix64(h + draw);
  return (double)(h >> 11) * (1.0 / 9007199254740992.0);
}
struct FGibbsArgs {
  uint64_t n_forests;
  const uint64_t* node_off;
  const uint32_t* next;
  const uint32_t* label;
  const uint8_t* backref;
  const uint32_t* norm;     // [rulespace] normalisation group or 0xFFFFFFFF (fixed probability = prior)
  const double* prior;
  double* count;            // sequential mode updates these between forests
  double* normsum;
  double* ins;              // [nodes] ln inside scratch
  const uint64_t* samp_base;
  const uint32_t* old_len;  // previous sample (removed first in sequential mode)
  const uint32_t* old_ids;
  uint32_t* new_len;
  uint32_t* new_ids;
  double power;
  uint64_t seed;
  uint32_t sweep;
  int sequential;
  int* err;
};
__device__ void forest_gibbs_one(const FGibbsArgs& A, uint64_t f) {
  const uint64_t base = A.node_off[f];
  const uint32_t n = (uint32_t)(A.node_off[f + 1] - base);
  const uint32_t* nx = A.next + base;
  const uint32_t* lb = A.label + base;
  const uint8_t* br = A.backref + base;
  double* in_ = A.ins + base;
  const uint64_t sb = A.samp_base[f];
  if (A.sequential) {  // addc(block, -wt): the forest's previous sample leaves the counts (gibbs.hpp:851-852)
    for (uint32_t k = 0, e = A.old_len[f]; k < e; ++k) {
      const uint32_t id = A.old_ids[sb + k], g = A.norm[id];
      if (g != 0xFFFFFFFFu) {
        A.count[id] -= 1.;
        A.normsum[g] -= 1.;
      }
    }
  }
  auto proposal_ln = [&](uint32_t id) -> double {
    const uint32_t g = A.norm[id];
    const double p = g != 0xFFFFFFFFu ? A.count[id] / A.normsum[g] : A.prior[id];
    return p > 0 ? log(p) : -CUDART_INF;
  };
  {  // compute_inside(W): post-order with a stack of open nodes
    uint32_t s_node[kGibbsDepth];
    double s_acc[kGibbsDepth];
    bool s_first[kGibbsDepth];
    int sp = 0;
    for (uint32_t i = 0; i < n; ++i) {
      double val = 0;
      bool done;
      if (br[i]) {
        val = in_[lb[i]];
        in_[i] = val;
        done = true;
      } else if (nx[i] == i + 1) {
        val = lb[i] ? proposal_ln(lb[i]) : -CUDART_INF;
        in_[i] = val;
        done = true;
      } else {
        if (sp >= kGibbsDepth) {
          *A.err = 1;
          return;
        }
        s_node[sp] = i;
        s_acc[sp] = lb[i] ? proposal_ln(lb[i]) : -CUDART_INF;
        s_first[sp] = true;
        ++sp;
        done = false;
      }
      while (done && sp > 0) {
        const int t = sp - 1;
        const uint32_t p = s_node[t];
        if (lb[p])
          s_acc[t] += val;  // AND: product
        else {
          s_acc[t] = s_first[t] ? val : ln_add<double>(s_acc[t], val);  // OR: first child, then += in order
          s_first[t] = false;
        }
        if (nx[p] == i + 1) {
          val = s_acc[t];
          in_[p] = val;
          --sp;
        } else
          done = false;
      }
    }
  }
  // choose_random: depth-first, children in order; the stack holds the nodes still to visit (bit 31: power 1)
  uint32_t st[kGibbsStack];
  int sp = 0;
  uint32_t len = 0, draw = 0;
  st[sp++] = 0u;
  while (sp > 0) {
    uint32_t b = st[--sp];
    const bool unit = (b >> 31) != 0;
    b &= 0x7fffffffu;
    const double power = unit ? 1. : A.power;
    if (br[b]) {
      st[sp++] = lb[b] | 0x80000000u;  // choose_random(l.pointer(), v): default power
      continue;
    }
    const uint32_t e = nx[b];
    if (lb[b] == 0) {
      double norm = -CUDART_INF;
      for (uint32_t i = b + 1; i != e; i = nx[i]) {
        const double x = in_[i];
        norm = ln_add<double>(norm, x > -CUDART_INF ? x * power : x);
      }
      uint32_t i = b + 1;
      double choice = fg_uniform(A.seed, A.sweep, (uint32_t)f, draw++);
      for (;;) {
        const double x = in_[i];
        choice -= exp((x > -CUDART_INF ? x * power : x) - norm);
        if (choice < 0) break;
        const uint32_t nn = nx[i];
        if (nn == e) break;
        i = nn;
      }
      st[sp++] = i | (unit ? 0x80000000u : 0u);
    } else {
      if (sb + len >= A.samp_base[f + 1]) {  // (a derivation that revisits shared sub-forests more often than budgeted)
        *A.err = 2;
        return;
      }
      A.new_ids[sb + len++] = lb[b];
      // children are pushed last to first so that the first child is visited next
      uint32_t cnt = 0;
      for (uint32_t c = b + 1; c < e; c = nx[c]) ++cnt;
      if (sp + (int)cnt > kGibbsStack) {
        *A.err = 1;
        return;
      }
      uint32_t k = 0;
      for (uint32_t c = b + 1; c < e; c = nx[c], ++k) st[sp + (cnt - 1 - k)] = c | (unit ? 0x80000000u : 0u);
      sp += (int)cnt;
    }
  }
  A.new_len[f] = len;
  if (A.sequential) {  // addc(block, +wt)
    for (uint32_t k = 0; k < len; ++k) {
      const uint32_t id = A.new_ids[sb + k], g = A.norm[id];
      if (g != 0xFFFFFFFFu) {
        A.count[id] += 1.;
        A.normsum[g] += 1.;
      }
    }
  }
}
__global__ void k_forest_gibbs_sequential(FGibbsArgs A) {  // the exact collapsed sampler: one thread walks the corpus
  if (blockIdx.x || threadIdx.x) return;
  for (uint64_t f = 0; f < A.n_forests; ++f) {
    forest_gibbs_one(A, f);
    if (*A.err) return;
  }
}
__global__ void k_forest_gibbs_batched(FGibbsArgs A) {  // every forest against the previous sweep's counts
  const uint64_t f = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (f < A.n_forests) forest_gibbs_one(A, f);
}
// batched mode: count deltas of the sweep (old sample out, new sample in)
__global__ void k_forest_gibbs_apply(uint64_t n_forests, const uint64_t* __restrict__ samp_base, const uint32_t* __restrict__ old_len,
                                     const uint32_t* __restrict__ old_ids, const uint32_t* __restrict__ new_len,
                                     const uint32_t* __restrict__ new_ids, const uint32_t* __restrict__ norm, double* count,
                                     double* normsum) {
  const uint64_t f = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (f >= n_forests) return;
  const uint64_t sb = samp_base[f];
  for (uint32_t k = 0, e = old_len[f]; k < e; ++k) {
    const uint32_t id = old_ids[sb + k], g = norm[id];
    if (g != 0xFFFFFFFFu) {
      atomicAdd(&count[id], -1.);
      atomicAdd(&normsum[g], -1.);
    }
  }
  for (uint32_t k = 0, e = new_len[f]; k < e; ++k) {
    const uint32_t id = new_ids[sb + k], g = norm[id];
    if (g != 0xFFFFFFFFu) {
      atomicAdd(&count[id], 1.);
      atomicAdd(&normsum[g], 1.);
    }
  }
}
__global__ void k_forest_gibbs_accumulate(uint64_t n, const double* __restrict__ count, double dt, double* __restrict__ cum) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) cum[i] += dt * count[i];
}

// counts := priors (restore_p0, gibbs.hpp:618-623); the forests stay on the device in the reference representation
extern "C" int cml_forests_gibbs_init(cml_forests* f, const cml_forest_batch* b, const cml_forest_gibbs_model* g) {
  if (!f || !b || !g || !g->param_norm || !g->param_prior) return CML_ERR_ARG;
  F_REQUIRE(f->have_rules, CML_ERR_STATE, "cml_forests_gibbs_init before cml_forests_set_rules");
  CML_CUDA(cudaSetDevice(f->device));
  cudaStream_t s = f->stream;
  const uint64_t nn = b->n_forests ? b->node_off[b->n_forests] : 0;
  std::vector<uint64_t> base(b->n_forests + 1, 0);
  for (uint64_t i = 0; i < b->n_forests; ++i) {
    uint64_t he = 0;
    for (uint64_t k = b->node_off[i]; k < b->node_off[i + 1]; ++k) he += (!b->backref[k] && b->label[k] != 0);
    // a shared sub-forest can be sampled through several references: bound the path by the node count of the forest
    base[i + 1] = base[i] + std::max<uint64_t>(he, b->node_off[i + 1] - b->node_off[i]) * 4;
  }
  for (uint64_t r = 0; r < f->rulespace; ++r)
    F_REQUIRE(g->param_norm[r] == 0xFFFFFFFFu || g->param_norm[r] < g->n_norms, CML_ERR_ARG, "param_norm out of range");
  f->g_forests = b->n_forests;
  f->g_nodes = nn;
  f->g_cap = base[b->n_forests];
  f->g_norms = g->n_norms;
  CML_CUDA(f->g_node_off.upload(b->node_off, b->n_forests + 1, s));
  CML_CUDA(f->g_next.upload(b->next, nn, s));
  CML_CUDA(f->g_label.upload(b->label, nn, s));
  CML_CUDA(f->g_backref.upload(b->backref, nn, s));
  CML_CUDA(f->g_samp_base.upload(base.data(), base.size(), s));
  CML_CUDA(f->g_norm.upload(g->param_norm, f->rulespace, s));
  CML_CUDA(f->g_prior.upload(g->param_prior, f->rulespace, s));
  CML_CUDA(f->g_count.upload(g->param_prior, f->rulespace, s));
  CML_CUDA(f->g_cum.alloc(f->rulespace));
  CML_CUDA(cudaMemsetAsync(f->g_cum.p, 0, f->rulespace * sizeof(double), s));
  std::vector<double> ns(std::max<uint32_t>(1, g->n_norms), 0.);
  for (uint64_t r = 0; r < f->rulespace; ++r)
    if (g->param_norm[r] != 0xFFFFFFFFu) ns[g->param_norm[r]] += g->param_prior[r];
  CML_CUDA(f->g_normsum.upload(ns.data(), ns.size(), s));
  CML_CUDA(f->g_ins.alloc(std::max<uint64_t>(1, nn)));
  for (int k = 0; k < 2; ++k) {
    CML_CUDA(f->g_sample[k].alloc(std::max<uint64_t>(1, f->g_cap)));
    CML_CUDA(f->g_len[k].alloc(std::max<uint64_t>(1, b->n_forests)));
    CML_CUDA(cudaMemsetAsync(f->g_len[k].p, 0, std::max<uint64_t>(1, b->n_forests) * sizeof(uint32_t), s));
  }
  CML_CUDA(f->g_err.alloc(1));
  CML_CUDA(cudaMemsetAsync(f->g_err.p, 0, sizeof(int), s));
  CML_CUDA(cudaStreamSynchronize(s));
  f->g_cur = 0;
  f->have_gibbs = true;
  return CML_OK;
}

// one sweep (gibbs_base::iteration): every forest resampled once; afterwards cum += accumulate_dt * count
extern "C" int cml_forests_gibbs_sweep(cml_forests* f, const cml_gibbs_sweep_opts* o) {
  if (!f || !o) return CML_ERR_ARG;
  F_REQUIRE(f->have_gibbs, CML_ERR_STATE, "cml_forests_gibbs_sweep before cml_forests_gibbs_init");
  CML_CUDA(cudaSetDevice(f->device));
  cudaStream_t s = f->stream;
  const int cur = f->g_cur, nxt = cur ^ 1;
  FGibbsArgs A;
  A.n_forests = f->g_forests;
  A.node_off = f->g_node_off.p;
  A.next = f->g_next.p;
  A.label = f->g_label.p;
  A.backref = f->g_backref.p;
  A.norm = f->g_norm.p;
  A.prior = f->g_prior.p;
  A.count = f->g_count.p;
  A.normsum = f->g_normsum.p;
  A.ins = f->g_ins.p;
  A.samp_base = f->g_samp_base.p;
  A.old_len = f->g_len[cur].p;
  A.old_ids = f->g_sample[cur].p;
  A.new_len = f->g_len[nxt].p;
  A.new_ids = f->g_sample[nxt].p;
  A.power = o->power;
  A.seed = o->seed;
  A.sweep = o->sweep;
  A.sequential = o->mode == CML_GIBBS_SEQUENTIAL;
  A.err = f->g_err.p;
  if (f->g_forests) {
    if (A.sequential) {
      k_forest_gibbs_sequential<<<1, 32, 0, s>>>(A);
      ++f->launches;
    } else {
      k_forest_gibbs_batched<<<f_cdiv(f->g_forests, 64), 64, 0, s>>>(A);
      k_forest_gibbs_apply<<<f_cdiv(f->g_forests, 128), 128, 0, s>>>(f->g_forests, f->g_samp_base.p, f->g_len[cur].p, f->g_sample[cur].p,
                                                                   f->g_len[nxt].p, f->g_sample[nxt].p, f->g_norm.p, f->g_count.p,
                                                                   f->g_normsum.p);
      f->launches += 2;
    }
  }
  if (o->accumulate_dt != 0.) {
    k_forest_gibbs_accumulate<<<f_cdiv(f->rulespace, 256), 256, 0, s>>>(f->rulespace, f->g_count.p, o->accumulate_dt, f->g_cum.p);
    ++f->launches;
  }
  CML_CUDA(cudaGetLastError());
  int herr = 0;
  CML_CUDA(cudaMemcpyAsync(&herr, f->g_err.p, sizeof(int), cudaMemcpyDeviceToHost, s));
  CML_CUDA(cudaStreamSynchronize(s));
  F_REQUIRE(!herr, CML_ERR_ARG,
            herr == 2 ? "cml_forests_gibbs_sweep: a sampled derivation is longer than its sample slot"
                      : "cml_forests_gibbs_sweep: a forest nests deeper than the sampler's stacks (96 levels)");
  f->g_cur = nxt;
  return CML_OK;
}
extern "C" uint64_t cml_forests_gibbs_sample_capacity(cml_forests* f) { return f ? f->g_cap : 0; }
// current sample: len[forest] rule ids at ids[base_f ..] in record order (choose_random's v.record), base_f from
// cml_forests_gibbs_sample_bases
extern "C" int cml_forests_gibbs_get_samples(cml_forests* f, uint32_t* len, uint32_t* ids, uint64_t cap, uint64_t* bases) {
  if (!f || !len || !ids) return CML_ERR_ARG;
  F_REQUIRE(f->have_gibbs && cap >= f->g_cap, CML_ERR_ARG, "cml_forests_gibbs_get_samples: no sampler state or buffer too small");
  CML_CUDA(cudaSetDevice(f->device));
  cudaStream_t s = f->stream;
  CML_CUDA(cudaMemcpyAsync(len, f->g_len[f->g_cur].p, f->g_forests * sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
  CML_CUDA(cudaMemcpyAsync(ids, f->g_sample[f->g_cur].p, f->g_cap * sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
  if (bases) CML_CUDA(cudaMemcpyAsync(bases, f->g_samp_base.p, (f->g_forests + 1) * sizeof(uint64_t), cudaMemcpyDeviceToHost, s));
  CML_CUDA(cudaStreamSynchronize(s));
  return CML_OK;
}
extern "C" int cml_forests_gibbs_get_state(cml_forests* f, double* count, double* cum, double* normsum) {
  if (!f) return CML_ERR_ARG;
  F_REQUIRE(f->have_gibbs, CML_ERR_STATE, "no sampler state");
  CML_CUDA(cudaSetDevice(f->device));
  cudaStream_t s = f->stream;
  if (count) CML_CUDA(cudaMemcpyAsync(count, f->g_count.p, f->rulespace * sizeof(double), cudaMemcpyDeviceToHost, s));
  if (cum) CML_CUDA(cudaMemcpyAsync(cum, f->g_cum.p, f->rulespace * sizeof(double), cudaMemcpyDeviceToHost, s));
  if (normsum) CML_CUDA(cudaMemcpyAsync(normsum, f->g_normsum.p, std::max<uint32_t>(1, f->g_norms) * sizeof(double), cudaMemcpyDeviceToHost, s));
  CML_CUDA(cudaStreamSynchronize(s));
  return CML_OK;
}
extern "C" int cml_forests_get_counts(cml_forests* f, double* counts, uint64_t n) {
  if (!f || !counts) return CML_ERR_ARG;
  F_REQUIRE(f->have_rules && n >= f->rulespace, CML_ERR_ARG, "cml_forests_get_counts: buffer too small");
  CML_CUDA(cudaSetDevice(f->device));
  CML_CUDA(cudaMemcpyAsync(counts, f->reduce.p, f->rulespace * sizeof(double), cudaMemcpyDeviceToHost, f->stream));
  CML_CUDA(cudaStreamSynchronize(f->stream));
  return CML_OK;
}
extern "C" int cml_forests_reduce_buffer(cml_forests* f, void** p, uint64_t* n) {
  if (!f || !p || !n) return CML_ERR_ARG;
  F_REQUIRE(f->have_rules, CML_ERR_STATE, "cml_forests_reduce_buffer before cml_forests_set_rules");
  *p = f->reduce.p;
  *n = f->rulespace + 3;
  return CML_OK;
}

static int forest_norm(cml_forests* f, const double* counts, double prior, double add_k, int zero_mode, double* max_delta,
                       uint64_t* max_index) {
  CML_CUDA(cudaSetDevice(f->device));
  if (f->n_groups) {
    k_forest_norm<<<f_cdiv(f->n_groups * 32, 256), 256, 0, f->stream>>>(f->n_groups, f->group_off.p, f->group_members.p, counts, prior,
                                                                     add_k, zero_mode, f->ln_w.p, f->gdiff.p, f->gidx.p);
    ++f->launches;
  }
  k_forest_maxdiff<<<1, 1024, 0, f->stream>>>(f->n_groups, f->gdiff.p, f->gidx.p, f->group_members.p, f->out_diff.p, f->out_rule.p);
  ++f->launches;
  CML_CUDA(cudaGetLastError());
  double d = 0;
  unsigned long long r = 0;
  CML_CUDA(cudaMemcpyAsync(&d, f->out_diff.p, sizeof(d), cudaMemcpyDeviceToHost, f->stream));
  CML_CUDA(cudaMemcpyAsync(&r, f->out_rule.p, sizeof(r), cudaMemcpyDeviceToHost, f->stream));
  CML_CUDA(cudaStreamSynchronize(f->stream));
  if (max_delta) *max_delta = d;
  if (max_index) *max_index = r;
  return CML_OK;
}
extern "C" int cml_forests_maximize(cml_forests* f, const cml_forest_norm_opts* o, double* max_delta, uint64_t* max_index) {
  if (!f || !o) return CML_ERR_ARG;
  F_REQUIRE(f->have_params, CML_ERR_STATE, "cml_forests_maximize before cml_forests_set_params");
  F_REQUIRE(!f->pending, CML_ERR_STATE, "cml_forests_maximize while an estimate is pending");
  return forest_norm(f, f->reduce.p, o->prior_total, o->add_k, o->zero_mode, max_delta, max_index);
}
extern "C" int cml_forests_normalize_params(cml_forests* f) {
  if (!f) return CML_ERR_ARG;
  F_REQUIRE(f->have_params, CML_ERR_STATE, "cml_forests_normalize_params before cml_forests_set_params");
  return forest_norm(f, nullptr, 0., 0., CML_FOREST_UNIFORM, nullptr, nullptr);
}

// ---------------------------------------------------------------------------------------------------
// host scaffold of the per-forest decoders (cml_forests_kbest, cml_forests_sample) over a batch as given to
// cml_forests_add: validation and levelisation, and the chunk plan
// ---------------------------------------------------------------------------------------------------
namespace {
struct ForestLevels {
  std::vector<uint32_t> order;     // per forest, at its node_off: its real nodes by height, then pre-order index
  std::vector<uint32_t> lvl;       // per forest, at lvl_base: n_levels + 1 offsets into its order
  std::vector<uint64_t> lvl_base;  // [n_forests + 1]
  uint32_t max_fanout = 0;         // the largest OR fan-out of the batch
  uint32_t max_levels = 0;         // levels of the tallest forest (a root-to-leaf path has at most this many real nodes)
};

// forest_pass1's heights, real nodes sorted by (height, pre-order index), on up to 32 host threads.  Errors name
// the entry point `who`: CML_ERR_ARG for an empty, too large or malformed forest or a rule id beyond rulespace,
// CML_ERR_CYCLE for a cyclic back reference (the first such forest is reported).
int forest_levelise(cml_forests* f, const cml_forest_batch* b, const char* who, ForestLevels& out) {
  const uint64_t nf = b->n_forests;
  for (uint64_t i = 0; i < nf; ++i) {
    F_REQUIRE(b->node_off[i] < b->node_off[i + 1], CML_ERR_ARG, std::string(who) + ": empty forest");
    F_REQUIRE(b->node_off[i + 1] - b->node_off[i] < 0x7fffffffull, CML_ERR_ARG, std::string(who) + ": forest too large");
  }
  const uint64_t n_nodes = b->node_off[nf];
  std::vector<FlatForest> ff(nf);
  std::vector<uint32_t> maxdeg(nf, 0);
  std::vector<std::vector<uint32_t>> lv(nf);
  out.order.assign(n_nodes, 0);
  std::vector<uint32_t>& order = out.order;
  {
    unsigned nt = std::max(1u, std::min(32u, std::thread::hardware_concurrency()));
    if (nf < 64) nt = 1;
    std::atomic<uint64_t> nextf(0);
    auto work = [&]() {
      ForestScratch S;
      for (;;) {
        const uint64_t i0 = nextf.fetch_add(64);
        if (i0 >= nf) break;
        for (uint64_t i = i0; i < std::min(nf, i0 + 64); ++i) {
          const uint64_t o = b->node_off[i];
          const uint32_t n = (uint32_t)(b->node_off[i + 1] - o);
          const uint32_t *nx = b->next + o, *lb = b->label + o;
          const uint8_t* br = b->backref + o;
          forest_pass1(n, nx, lb, br, f->rulespace, S, ff[i]);
          if (ff[i].error) continue;
          std::vector<uint32_t>& L = lv[i];
          L.assign(ff[i].n_levels + 1, 0);
          for (uint32_t p = 0; p < n; ++p)
            if (!br[p]) {
              ++L[S.height[p] + 1];
              if (!lb[p]) {
                uint32_t m = 0;
                for (uint32_t q = p + 1; q < nx[p]; q = nx[q]) ++m;
                maxdeg[i] = std::max(maxdeg[i], m);
              }
            }
          for (uint32_t h = 0; h < ff[i].n_levels; ++h) L[h + 1] += L[h];
          S.cnt.assign(L.begin(), L.end() - 1);
          for (uint32_t p = 0; p < n; ++p)
            if (!br[p]) order[o + S.cnt[S.height[p]]++] = p;
        }
      }
    };
    std::vector<std::thread> th;
    for (unsigned t = 1; t < nt; ++t) th.emplace_back(work);
    work();
    for (auto& t : th) t.join();
  }
  out.lvl_base.assign(nf + 1, 0);
  out.max_fanout = out.max_levels = 0;
  for (uint64_t i = 0; i < nf; ++i) {
    if (ff[i].error) {
      f->err = std::string(who) + ": forest " + std::to_string(i) +
               (ff[i].error == 2 ? " has a cyclic back reference" : ff[i].error == 3 ? " uses a rule id beyond rulespace" : " is malformed");
      return ff[i].error == 2 ? CML_ERR_CYCLE : CML_ERR_ARG;
    }
    out.lvl_base[i + 1] = out.lvl_base[i] + lv[i].size();
    out.max_fanout = std::max(out.max_fanout, maxdeg[i]);
    out.max_levels = std::max(out.max_levels, ff[i].n_levels);
  }
  out.lvl.assign(out.lvl_base[nf], 0);
  for (uint64_t i = 0; i < nf; ++i) std::copy(lv[i].begin(), lv[i].end(), out.lvl.begin() + out.lvl_base[i]);
  return CML_OK;
}

// chunks of consecutive forests whose scratch (per_node bytes per pre-order node, per_forest per forest) fits the
// budget; a larger forest gets a chunk of its own
struct ForestChunks {
  std::vector<uint64_t> begin;  // chunk c is forests [begin[c], begin[c + 1])
  uint64_t max_nodes = 0, max_forests = 0;
};
ForestChunks forest_chunks(const cml_forest_batch* b, uint64_t per_node, uint64_t per_forest, uint64_t budget) {
  const uint64_t nf = b->n_forests;
  ForestChunks P;
  P.begin.assign(1, 0);
  for (uint64_t i = 0; i < nf; ++i) {
    const uint64_t c0 = P.begin.back();
    if (i > c0 && (b->node_off[i + 1] - b->node_off[c0]) * per_node + (i + 1 - c0) * per_forest > budget) P.begin.push_back(i);
  }
  P.begin.push_back(nf);
  for (size_t c = 0; c + 1 < P.begin.size(); ++c) {
    P.max_nodes = std::max(P.max_nodes, b->node_off[P.begin[c + 1]] - b->node_off[P.begin[c]]);
    P.max_forests = std::max(P.max_forests, P.begin[c + 1] - P.begin[c]);
  }
  return P;
}
}  // namespace

// ---------------------------------------------------------------------------------------------------
// k best derivations of every forest (forest-em -v --kbest=n): an eager k-best merge over the hypergraph, bottom-up by
// height.  A derivation is a choice of one child at every OR node it reaches; a shared node (back reference) is
// expanded independently at every use.  Lists are best first, with a fixed tie key:
//   OR node     top k over its children's entries: score desc, then child pre-order position, then child rank;
//   AND node    rule weight w, slots s1..sm: a left fold  L0 = [w],  Lj = top k { L(j-1)[a] + sj[b] }, ties by a then b
//               (the sums in k_forest_viterbi's order, so rank 0 is its derivation, bit for bit);
//   back ref.   its shared node's list.
// Every list entry carries its score, a back pointer -- OR: (resolved child node, its rank); fold: (a, b) -- and the
// size of its subtree in AND nodes (1 + the slots' sizes for AND, the chosen child's size for OR), so the output offsets
// of a derivation's nodes are known without walking it: extraction needs no stack and no depth limit.
//
// k_forest_kbest: one warp per forest.  Real nodes come levelised by height (forest_pass1's heights, which already see
// through back references); the nodes of one height never feed each other and are merged in parallel by lane groups of
// G lanes, heights are separated by __syncwarp.  A merge is k rounds of a shuffle arg-max over the group; lane g owns
// candidate rows g, g + G, ... (OR: one head per child; fold: one cursor per entry of L(j-1), rows opened one at a time --
// row a + 1 cannot win before row a has given its first entry) and keeps its best head in registers, its rows' cursors
// in a per-group scratch.  Lists live in global memory (a chunk's scratch).
// k_forest_kbest_paths: one thread per derivation writes its AND nodes in pre-order: a node at offset o puts slot j's
// node at o + size(L(j-1)[a]) (L0: o + 1), so every position is filled before the walk reaches it.
// ---------------------------------------------------------------------------------------------------
namespace {
const uint32_t kFkNone = 0xFFFFFFFFu;
const int kFkWarps = 4;  // warps per block
struct FkArgs {
  const uint64_t* node_off;  // [n_forests + 1] the batch's pre-order arrays
  const uint32_t* next;
  const uint32_t* label;
  const uint8_t* backref;
  const uint32_t* order;     // per forest, at its node_off: its real nodes by height, then pre-order index
  const uint32_t* lvl;       // per forest, at lvl_base: n_levels + 1 offsets into its order
  const uint64_t* lvl_base;  // [n_forests + 1]
  const double* ln_w;
  uint64_t f0, s0;           // first forest of the chunk and its first node (chunk-local node = batch node - s0)
  uint32_t n_f, k;
  // per chunk-local pre-order node: its own list (x*) and, for a child slot of an AND node, the fold through it (f*)
  double* xs;
  uint2* xb;
  uint32_t *xz, *xl;
  double* fs;
  uint2* fb;
  uint32_t *fz, *fl;
  uint32_t* prv;   // child slot of an AND node -> the previous slot (kFkNone: the first)
  uint32_t* lst;   // AND node with children -> its last slot
  uint2* cur;      // per lane group: cstride (child node, cursor) rows
  uint32_t cstride;
  double* score;   // [n_f * k] this chunk's results
  uint32_t* n_and;
};

__device__ __forceinline__ uint32_t fk_sat(uint32_t a, uint32_t b) {  // subtree sizes saturate at kFkNone
  const uint32_t s = a + b;
  return s < a ? kFkNone : s;
}

template <int G>
__device__ __forceinline__ void fk_argmax(unsigned gmask, double& v, uint32_t& q) {  // score desc, then row asc
#pragma unroll
  for (int o = G / 2; o > 0; o >>= 1) {
    const double ov = __shfl_xor_sync(gmask, v, o, G);
    const uint32_t oq = __shfl_xor_sync(gmask, q, o, G);
    if (ov > v || (ov == v && oq < q)) {
      v = ov;
      q = oq;
    }
  }
}

// Lj = top k { P[a] + S[b] } (ties by a, then b) into (os, ob, oz); returns its length
template <int G>
__device__ __forceinline__ uint32_t fk_fold(unsigned gmask, uint32_t g, uint32_t k, const double* __restrict__ ps, const uint32_t* __restrict__ pz,
                            uint32_t la, const double* __restrict__ cs, const uint32_t* __restrict__ cz, uint32_t lc,
                            double* __restrict__ os, uint2* __restrict__ ob, uint32_t* __restrict__ oz, uint2* __restrict__ C) {
  if (!la || !lc) return 0;
  uint32_t act = 1;  // open rows
  if (g == 0) C[0].y = 0;
  double bv = g == 0 ? ps[0] + cs[0] : -CUDART_INF;
  uint32_t ba = g == 0 ? 0u : kFkNone;
  uint32_t r = 0;
  for (; r < k; ++r) {
    double v = bv;
    uint32_t a = ba;
    fk_argmax<G>(gmask, v, a);
    if (!(v > -CUDART_INF)) break;  // group-uniform: no candidate left
    const bool opened = a + 1 == act && act < la;
    if (opened) ++act;
    const bool mine = a % G == g, gets_row = opened && (act - 1) % G == g;
    if (mine) {
      const uint32_t c0 = C[a].y;
      os[r] = v;
      ob[r] = make_uint2(a, c0);
      oz[r] = fk_sat(pz[a], cz[c0]);
      C[a].y = c0 + 1;
    }
    if (gets_row) C[act - 1].y = 0;
    if (mine || gets_row) {
      bv = -CUDART_INF;
      ba = kFkNone;
      for (uint32_t q = g; q < act; q += G) {
        const uint32_t c = C[q].y;
        if (c < lc) {
          const double h = ps[q] + cs[c];
          if (h > bv) {
            bv = h;
            ba = q;
          }
        }
      }
    }
  }
  return r;
}

template <int G>
__global__ void __launch_bounds__(kFkWarps * 32, 1) k_forest_kbest(FkArgs A) {
  const uint32_t lane = threadIdx.x & 31, g = lane % G, grp = lane / G;
  const unsigned gmask = G == 32 ? 0xFFFFFFFFu : (((1u << G) - 1u) << (grp * G));
  const uint32_t k = A.k;
  const uint32_t gw = blockIdx.x * kFkWarps + threadIdx.x / 32, nw = gridDim.x * kFkWarps;
  uint2* __restrict__ C = A.cur + ((uint64_t)gw * (32 / G) + grp) * A.cstride;
  for (uint32_t w = gw; w < A.n_f; w += nw) {
    const uint64_t f = A.f0 + w, nb = A.node_off[f], sb = nb - A.s0;
    const uint32_t* __restrict__ nx = A.next + nb;
    const uint32_t* __restrict__ lb = A.label + nb;
    const uint8_t* __restrict__ br = A.backref + nb;
    const uint32_t* __restrict__ ord = A.order + nb;
    const uint32_t* __restrict__ lv = A.lvl + A.lvl_base[f];
    const uint32_t nl = (uint32_t)(A.lvl_base[f + 1] - A.lvl_base[f]) - 1;
    double* __restrict__ XS = A.xs + sb * k;
    uint2* __restrict__ XB = A.xb + sb * k;
    uint32_t* __restrict__ XZ = A.xz + sb * k;
    uint32_t* __restrict__ XL = A.xl + sb;
    double* __restrict__ FS = A.fs + sb * k;
    uint2* __restrict__ FB = A.fb + sb * k;
    uint32_t* __restrict__ FZ = A.fz + sb * k;
    uint32_t* __restrict__ FL = A.fl + sb;
    for (uint32_t l = 0; l < nl; ++l) {
      const uint32_t j1 = lv[l + 1];
      for (uint32_t j = lv[l] + grp; j < j1; j += 32 / G) {  // group-uniform
        const uint32_t p = ord[j], e = nx[p], lab = lb[p];
        if (lab) {  // AND node
          const double wv = A.ln_w[lab];
          if (e == p + 1) {  // a leaf rule
            if (g == 0) {
              const bool ok = wv > -CUDART_INF;
              if (ok) {
                XS[(uint64_t)p * k] = wv;
                XB[(uint64_t)p * k] = make_uint2(0, 0);
                XZ[(uint64_t)p * k] = 1;
              }
              XL[p] = ok ? 1 : 0;
            }
            continue;
          }
          uint32_t prev = kFkNone;
          for (uint32_t b = p + 1; b < e;) {
            const uint32_t c = br[b] ? lb[b] : b, b1 = nx[b];
            const bool last = b1 >= e;
            const uint64_t o = (uint64_t)(last ? p : b) * k;
            double* os = (last ? XS : FS) + o;
            uint2* ob = (last ? XB : FB) + o;
            uint32_t* oz = (last ? XZ : FZ) + o;
            const double* cs = XS + (uint64_t)c * k;
            const uint32_t* cz = XZ + (uint64_t)c * k;
            const uint32_t lc = XL[c];
            uint32_t len;
            if (prev == kFkNone) {  // L1 = [w] + s1: the slot's list shifted by the rule weight
              len = wv > -CUDART_INF ? min(k, lc) : 0u;
              for (uint32_t r = g; r < len; r += G) {
                os[r] = wv + cs[r];
                ob[r] = make_uint2(0, r);
                oz[r] = fk_sat(1u, cz[r]);
              }
            } else {
              len = fk_fold<G>(gmask, g, k, FS + (uint64_t)prev * k, FZ + (uint64_t)prev * k, FL[prev], cs, cz, lc, os, ob, oz, C);
            }
            if (g == 0) {
              (last ? XL[p] : FL[b]) = len;
              A.prv[sb + b] = prev;
            }
            __syncwarp(gmask);  // the next fold reads this one
            prev = b;
            b = b1;
          }
          if (g == 0) A.lst[sb + p] = prev;
        } else {  // OR node: merge of the children's lists, one head per child
          double bv = -CUDART_INF;
          uint32_t bq = kFkNone, m = 0;
          for (uint32_t b = p + 1; b < e; b = nx[b], ++m)
            if (m % G == g) {
              const uint32_t c = br[b] ? lb[b] : b;
              C[m] = make_uint2(c, 0);
              if (XL[c] && XS[(uint64_t)c * k] > bv) {
                bv = XS[(uint64_t)c * k];
                bq = m;
              }
            }
          double* os = XS + (uint64_t)p * k;
          uint2* ob = XB + (uint64_t)p * k;
          uint32_t* oz = XZ + (uint64_t)p * k;
          uint32_t r = 0;
          for (; r < k; ++r) {
            double v = bv;
            uint32_t q = bq;
            fk_argmax<G>(gmask, v, q);
            if (!(v > -CUDART_INF)) break;
            if (q % G == g) {  // the owner appends the winner, advances that child's cursor and rescans its rows
              const uint2 cc = C[q];
              os[r] = v;
              ob[r] = cc;
              oz[r] = XZ[(uint64_t)cc.x * k + cc.y];
              C[q].y = cc.y + 1;
              bv = -CUDART_INF;
              bq = kFkNone;
              for (uint32_t t = g; t < m; t += G) {
                const uint2 d = C[t];
                if (d.y < XL[d.x]) {
                  const double h = XS[(uint64_t)d.x * k + d.y];
                  if (h > bv) {
                    bv = h;
                    bq = t;
                  }
                }
              }
            }
          }
          if (g == 0) XL[p] = r;
        }
      }
      __syncwarp();
    }
    const uint32_t L0 = XL[0];  // the root
    for (uint32_t r = lane; r < k; r += 32) {
      A.score[(uint64_t)w * k + r] = r < L0 ? XS[r] : -CUDART_INF;
      A.n_and[(uint64_t)w * k + r] = r < L0 ? XZ[r] : 0u;
    }
    __syncwarp();
  }
}

// derivation t = (chunk forest t / k, rank t % k): its AND nodes (in-forest pre-order indices) at out[obase[t] ..]
__global__ void k_forest_kbest_paths(FkArgs A, const uint64_t* __restrict__ obase, uint32_t* __restrict__ out,
                                     uint32_t* __restrict__ orank) {
  const uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const uint32_t k = A.k;
  if (t >= (uint64_t)A.n_f * k) return;
  const uint32_t n = A.n_and[t];
  if (!n) return;
  const uint64_t f = A.f0 + t / k, nb = A.node_off[f], sb = nb - A.s0;
  const uint32_t* __restrict__ nx = A.next + nb;
  const uint32_t* __restrict__ lb = A.label + nb;
  const uint8_t* __restrict__ br = A.backref + nb;
  const uint2* __restrict__ XB = A.xb + sb * k;
  const uint2* __restrict__ FB = A.fb + sb * k;
  const uint32_t* __restrict__ FZ = A.fz + sb * k;
  const uint32_t* __restrict__ prv = A.prv + sb;
  const uint32_t* __restrict__ lst = A.lst + sb;
  uint32_t* __restrict__ o = out + obase[t];
  uint32_t* __restrict__ rk = orank + obase[t];
  auto put = [&](uint32_t c, uint32_t r, uint32_t at) {  // real node c's rank r, down to the AND node it stands for
    while (!lb[c]) {
      const uint2 x = XB[(uint64_t)c * k + r];
      c = x.x;
      r = x.y;
    }
    o[at] = c;
    rk[at] = r;
  };
  put(0, (uint32_t)(t % k), 0);
  for (uint32_t i = 0; i < n; ++i) {
    const uint32_t p = o[i];
    if (nx[p] == p + 1) continue;
    uint32_t j = lst[p];
    uint2 bp = XB[(uint64_t)p * k + rk[i]];  // the last fold is the node's own list
    for (;;) {  // the slots, last to first
      const uint32_t pj = prv[j];
      put(br[j] ? lb[j] : j, bp.y, i + (pj == kFkNone ? 1u : FZ[(uint64_t)pj * k + bp.x]));
      if (pj == kFkNone) break;
      bp = FB[(uint64_t)pj * k + bp.x];
      j = pj;
    }
  }
}
}  // namespace

extern "C" int cml_forests_set_kbest_scratch_mb(cml_forests* f, uint64_t mb) {
  if (!f) return CML_ERR_ARG;
  F_REQUIRE(mb > 0, CML_ERR_ARG, "cml_forests_set_kbest_scratch_mb: the budget must be at least 1 MiB");
  f->kbest_scratch_mb = mb;
  return CML_OK;
}

extern "C" int cml_forests_kbest_stats(cml_forests* f, uint64_t* scratch_bytes, uint64_t* chunks, float* kernel_ms) {
  if (!f) return CML_ERR_ARG;
  if (scratch_bytes) *scratch_bytes = f->kbest_scratch;
  if (chunks) *chunks = f->kbest_chunks;
  if (kernel_ms) *kernel_ms = f->kbest_ms;
  return CML_OK;
}

extern "C" int cml_forests_kbest(cml_forests* f, const cml_forest_batch* b, uint32_t k, double* ln_score, uint32_t* n_and,
                                 uint64_t* base, uint32_t* nodes, uint64_t cap) {
  if (!f || !b || !ln_score || !n_and || !base) return CML_ERR_ARG;
  F_REQUIRE(f->have_params, CML_ERR_STATE, "cml_forests_kbest before cml_forests_set_params");
  F_REQUIRE(k > 0, CML_ERR_ARG, "cml_forests_kbest: k must be at least 1");
  const uint64_t nf = b->n_forests;
  F_REQUIRE(nf == 0 || (b->node_off && b->next && b->label && b->backref), CML_ERR_ARG, "cml_forests_kbest: null array");
  CML_CUDA(cudaSetDevice(f->device));
  f->kbest_ms = 0;
  f->kbest_scratch = 0;
  f->kbest_chunks = 0;
  base[0] = 0;
  if (!nf) return CML_OK;
  ForestLevels L;
  if (const int rc = forest_levelise(f, b, "cml_forests_kbest", L)) return rc;
  const uint64_t n_nodes = b->node_off[nf];
  std::vector<uint32_t>& order = L.order;
  std::vector<uint32_t>& lvl = L.lvl;
  std::vector<uint64_t>& lvl_base = L.lvl_base;
  const uint32_t cstride = std::max(k, L.max_fanout);
  const uint64_t per_node = 40ull * k + 16;
  const ForestChunks P = forest_chunks(b, per_node, 0, f->kbest_scratch_mb << 20);
  const std::vector<uint64_t>& chunk = P.begin;
  const uint64_t n_chunks = chunk.size() - 1, max_nodes = P.max_nodes, max_forests = P.max_forests;
  cudaStream_t s = f->stream;
  const int G = k > 16 ? 32 : 8;
  const unsigned max_blocks = (unsigned)f->sm_count * 16u;
  const unsigned grid_cap = std::max(1u, std::min(f_cdiv(max_forests, kFkWarps), max_blocks));
  const uint64_t n_groups = (uint64_t)grid_cap * kFkWarps * (32 / G);
  DevArray<uint64_t> d_off, d_lvlb, d_obase;
  DevArray<uint32_t> d_next, d_label, d_order, d_lvl, d_xz, d_xl, d_fz, d_fl, d_prv, d_lst, d_nand, d_out, d_rank;
  DevArray<uint8_t> d_br;
  DevArray<double> d_xs, d_fs, d_score;
  DevArray<uint2> d_xb, d_fb, d_cur;
  CML_CUDA(d_off.upload(b->node_off, nf + 1, s));
  CML_CUDA(d_next.upload(b->next, n_nodes, s));
  CML_CUDA(d_label.upload(b->label, n_nodes, s));
  CML_CUDA(d_br.upload(b->backref, n_nodes, s));
  CML_CUDA(d_order.upload(order.data(), n_nodes, s));
  CML_CUDA(d_lvl.upload(lvl.data(), lvl.size(), s));
  CML_CUDA(d_lvlb.upload(lvl_base.data(), nf + 1, s));
  CML_CUDA(d_xs.alloc(max_nodes * k));
  CML_CUDA(d_xb.alloc(max_nodes * k));
  CML_CUDA(d_xz.alloc(max_nodes * k));
  CML_CUDA(d_xl.alloc(max_nodes));
  CML_CUDA(d_fs.alloc(max_nodes * k));
  CML_CUDA(d_fb.alloc(max_nodes * k));
  CML_CUDA(d_fz.alloc(max_nodes * k));
  CML_CUDA(d_fl.alloc(max_nodes));
  CML_CUDA(d_prv.alloc(max_nodes));
  CML_CUDA(d_lst.alloc(max_nodes));
  CML_CUDA(d_cur.alloc(n_groups * cstride));
  CML_CUDA(d_score.alloc(max_forests * k));
  CML_CUDA(d_nand.alloc(max_forests * k));
  CML_CUDA(d_obase.alloc(max_forests * k));
  f->kbest_chunks = n_chunks;
  f->kbest_scratch = max_nodes * per_node + n_groups * cstride * sizeof(uint2);
  FkArgs A{d_off.p, d_next.p, d_label.p, d_br.p, d_order.p, d_lvl.p, d_lvlb.p, f->ln_w.p, 0, 0, 0, k,
           d_xs.p, d_xb.p, d_xz.p, d_xl.p, d_fs.p, d_fb.p, d_fz.p, d_fl.p, d_prv.p, d_lst.p, d_cur.p, cstride,
           d_score.p, d_nand.p};
  EventPair ev, ev_paths;  // k_forest_kbest, k_forest_kbest_paths
  CML_CUDA(ev.create());
  CML_CUDA(ev_paths.create());
  bool fits = true, too_big = false;
  std::vector<uint64_t> obase;
  for (uint64_t c = 0; c < n_chunks; ++c) {
    const uint64_t f0 = chunk[c], nfc = chunk[c + 1] - f0, e0 = f0 * k, ne = nfc * k;
    A.f0 = f0;
    A.s0 = b->node_off[f0];
    A.n_f = (uint32_t)nfc;
    const unsigned grid = std::max(1u, std::min(f_cdiv(nfc, kFkWarps), grid_cap));
    CML_CUDA(cudaEventRecord(ev.a, s));
    if (G == 32)
      k_forest_kbest<32><<<grid, kFkWarps * 32, 0, s>>>(A);
    else
      k_forest_kbest<8><<<grid, kFkWarps * 32, 0, s>>>(A);
    ++f->launches;
    CML_CUDA(cudaGetLastError());
    CML_CUDA(cudaEventRecord(ev.b, s));
    CML_CUDA(cudaMemcpyAsync(ln_score + e0, d_score.p, ne * sizeof(double), cudaMemcpyDeviceToHost, s));
    CML_CUDA(cudaMemcpyAsync(n_and + e0, d_nand.p, ne * sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
    CML_CUDA(cudaStreamSynchronize(s));
    float ms = 0;
    CML_CUDA(cudaEventElapsedTime(&ms, ev.a, ev.b));
    f->kbest_ms += ms;
    obase.resize(ne);
    for (uint64_t i = 0; i < ne; ++i) {
      obase[i] = base[e0 + i] - base[e0];
      too_big |= n_and[e0 + i] == kFkNone;
      base[e0 + i + 1] = base[e0 + i] + n_and[e0 + i];
    }
    const uint64_t total = base[e0 + ne] - base[e0];
    fits = fits && !too_big && (!nodes || base[e0 + ne] <= cap);
    if (!nodes || !fits || !total) continue;
    if (d_out.n < total) {
      CML_CUDA(d_out.alloc(total));
      CML_CUDA(d_rank.alloc(total));
    }
    CML_CUDA(cudaMemcpyAsync(d_obase.p, obase.data(), ne * sizeof(uint64_t), cudaMemcpyHostToDevice, s));
    CML_CUDA(cudaEventRecord(ev_paths.a, s));
    k_forest_kbest_paths<<<f_cdiv(ne, 256), 256, 0, s>>>(A, d_obase.p, d_out.p, d_rank.p);
    ++f->launches;
    CML_CUDA(cudaGetLastError());
    CML_CUDA(cudaEventRecord(ev_paths.b, s));
    CML_CUDA(cudaMemcpyAsync(nodes + base[e0], d_out.p, total * sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
    CML_CUDA(cudaStreamSynchronize(s));
    CML_CUDA(cudaEventElapsedTime(&ms, ev_paths.a, ev_paths.b));
    f->kbest_ms += ms;
  }
  F_REQUIRE(!too_big, CML_ERR_ARG, "cml_forests_kbest: a derivation has more than 2^32 - 2 AND nodes");
  F_REQUIRE(!nodes || base[nf * k] <= cap, CML_ERR_ARG,
            "cml_forests_kbest: nodes buffer too small (need base[n_forests * k] = " + std::to_string(base[nf * k]) + ")");
  return CML_OK;
}

// ---------------------------------------------------------------------------------------------------
// The total weight of every forest, and derivations drawn in proportion to their weight (forest-em -v FILE --sample=n):
// the pre-order walk of FForest::choose_random (forest-em/forest.hpp:726-758) at fixed weights, on counter-based
// uniforms, so a draw does not depend on the launch shape, the chunking or the other forests.
//
// k_forest_sample: one warp per forest.  First an inside pass over the real nodes by height (the levelisation of
// cml_forests_kbest; the nodes of one height never feed each other, so they are spread over the lanes, and heights are
// separated by __syncwarp): in(AND) = ln_w[rule] + in(s1) + ... + in(sm) in slot order, in(OR) = a max-shifted
// log-sum-exp over the children in order, next to the saturating size of the node's largest derivation of non-zero
// weight.  Then lane j draws samples j, j + 32, ...  A walk records every AND node it reaches and draws one uniform per
// OR node; it keeps one (next slot, end of slots) entry for every AND node on the current path with slots still to
// visit.  The real nodes of a path have strictly falling heights, so a walker's stack holds at most n_levels entries;
// the stacks live in a chunk scratch of n_levels of the tallest forest per walker.
// k_forest_sample_paths: one thread per sample walks it again with the same uniforms and writes its AND nodes.
// ---------------------------------------------------------------------------------------------------
namespace {
const int kFsWarps = 4;  // warps per block of k_forest_sample; k_forest_sample_paths runs kFsWarps * 32 threads a block
struct FsArgs {
  const uint64_t* node_off;  // [n_forests + 1] the batch's pre-order arrays
  const uint32_t* next;
  const uint32_t* label;
  const uint8_t* backref;
  const uint32_t* order;     // per forest, at its node_off: its real nodes by height, then pre-order index
  const uint32_t* lvl;       // per forest, at lvl_base: n_levels + 1 offsets into its order
  const uint64_t* lvl_base;  // [n_forests + 1]
  const double* ln_w;
  const uint64_t* key;       // [n_forests] the key of forest i's uniforms, or null (key = i)
  uint64_t seed;
  uint64_t f0, s0;           // first forest of the chunk and its first node (chunk-local node = batch node - s0)
  uint32_t n_f, n;
  double* ins;               // [chunk-local pre-order node] inside value of a real node
  uint32_t* big;             // [chunk-local pre-order node] AND nodes of its largest derivation of non-zero weight
  uint2* stack;              // [walker * stride] (next slot, end of the slots) of an AND node on the walk's path
  uint32_t stride;
  double* ln_total;          // [n_f] this chunk's results
  double* ln_weight;         // [n_f * n]
  uint32_t* n_and;           // [n_f * n]
};

// sample r of chunk forest w: returns its number of AND nodes and sets wsum to the sum of their rules' ln weights, in
// pre-order; with out != null also writes the nodes (in-forest pre-order indices)
__device__ uint32_t fs_walk(const FsArgs& A, uint32_t w, uint32_t r, uint2* __restrict__ st, double& wsum,
                            uint32_t* __restrict__ out) {
  const uint64_t f = A.f0 + w, nb = A.node_off[f];
  const uint32_t* __restrict__ nx = A.next + nb;
  const uint32_t* __restrict__ lb = A.label + nb;
  const uint8_t* __restrict__ br = A.backref + nb;
  const double* __restrict__ I = A.ins + (nb - A.s0);
  const uint64_t h0 = mix64(A.seed ^ mix64(A.key ? A.key[f] : f));
  uint32_t c = 0, t = 0, m = 0, depth = 0;
  double ws = 0.;
  for (;;) {
    while (!lb[c]) {  // OR node (in(c) > -inf): the first child after which u - p_1 - ... - p_j < 0
      double u = sample_uniform(h0, r, t++);
      const double ic = I[c];
      uint32_t pick = kFkNone, last = kFkNone;
      for (uint32_t b = c + 1; b < nx[c]; b = nx[b]) {
        const uint32_t d = br[b] ? lb[b] : b;
        const double p = exp(I[d] - ic);
        if (p > 0.) {
          last = d;
          u -= p;
          if (u < 0.) {
            pick = d;
            break;
          }
        }
      }
      c = pick != kFkNone ? pick : last;  // rounding left u >= 0: the last child that can be taken
    }
    if (out) out[m] = c;
    ++m;
    ws += A.ln_w[lb[c]];
    const uint32_t e = nx[c];
    uint32_t b;
    if (e > c + 1) {  // its first slot next, the others pending
      b = c + 1;
      if (nx[b] < e) st[depth++] = make_uint2(nx[b], e);
    } else {  // a leaf rule: the next slot of the innermost AND node with one left
      if (!depth) break;
      const uint2 top = st[depth - 1];
      b = top.x;
      if (nx[b] < top.y)
        st[depth - 1].x = nx[b];
      else
        --depth;
    }
    c = br[b] ? lb[b] : b;
  }
  wsum = ws;
  return m;
}

__global__ void __launch_bounds__(kFsWarps * 32) k_forest_sample(FsArgs A) {
  const uint32_t lane = threadIdx.x & 31;
  const uint32_t gw = blockIdx.x * kFsWarps + threadIdx.x / 32, nw = gridDim.x * kFsWarps;
  uint2* __restrict__ st = A.stack + ((uint64_t)gw * 32 + lane) * A.stride;
  for (uint32_t w = gw; w < A.n_f; w += nw) {
    const uint64_t f = A.f0 + w, nb = A.node_off[f], sb = nb - A.s0;
    const uint32_t* __restrict__ nx = A.next + nb;
    const uint32_t* __restrict__ lb = A.label + nb;
    const uint8_t* __restrict__ br = A.backref + nb;
    const uint32_t* __restrict__ ord = A.order + nb;
    const uint32_t* __restrict__ lv = A.lvl + A.lvl_base[f];
    const uint32_t nl = (uint32_t)(A.lvl_base[f + 1] - A.lvl_base[f]) - 1;
    double* __restrict__ I = A.ins + sb;
    uint32_t* __restrict__ Z = A.big + sb;
    for (uint32_t l = 0; l < nl; ++l) {
      for (uint32_t j = lv[l] + lane; j < lv[l + 1]; j += 32) {
        const uint32_t p = ord[j], e = nx[p], lab = lb[p];
        double v;
        uint32_t z = 0;
        if (lab) {  // AND node: the rule, then the slots in order
          v = A.ln_w[lab];
          z = 1;
          for (uint32_t b = p + 1; b < e; b = nx[b]) {
            const uint32_t d = br[b] ? lb[b] : b;
            v = v + I[d];
            z = fk_sat(z, Z[d]);
          }
          if (!(v > -CUDART_INF)) z = 0;
        } else {  // OR node
          double mx = -CUDART_INF;
          for (uint32_t b = p + 1; b < e; b = nx[b]) {
            const uint32_t d = br[b] ? lb[b] : b;
            mx = fmax(mx, I[d]);
            if (I[d] > -CUDART_INF) z = max(z, Z[d]);
          }
          if (mx > -CUDART_INF) {
            double sum = 0.;
            for (uint32_t b = p + 1; b < e; b = nx[b]) sum += exp(I[br[b] ? lb[b] : b] - mx);
            v = mx + log(sum);
          } else {
            v = -CUDART_INF;
          }
        }
        I[p] = v;
        Z[p] = z;
      }
      __syncwarp();
    }
    const double total = I[0];
    const bool too_big = Z[0] == kFkNone;  // refused: no draw starts
    if (lane == 0) A.ln_total[w] = total;
    for (uint32_t r = lane; r < A.n; r += 32) {
      const uint64_t o = (uint64_t)w * A.n + r;
      if (!(total > -CUDART_INF) || too_big) {
        A.ln_weight[o] = -CUDART_INF;
        A.n_and[o] = too_big ? kFkNone : 0u;
        continue;
      }
      double ws;
      A.n_and[o] = fs_walk(A, w, r, st, ws, nullptr);
      A.ln_weight[o] = ws;
    }
    __syncwarp();
  }
}

// sample t = (chunk forest t / n, sample t % n): its AND nodes at out[obase[t] ..]
__global__ void __launch_bounds__(kFsWarps * 32) k_forest_sample_paths(FsArgs A, const uint64_t* __restrict__ obase,
                                                                       uint32_t* __restrict__ out) {
  const uint64_t g = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x, ng = (uint64_t)gridDim.x * blockDim.x;
  uint2* __restrict__ st = A.stack + g * A.stride;
  for (uint64_t t = g; t < (uint64_t)A.n_f * A.n; t += ng) {
    if (!A.n_and[t]) continue;
    double ws;
    fs_walk(A, (uint32_t)(t / A.n), (uint32_t)(t % A.n), st, ws, out + obase[t]);
  }
}
}  // namespace

extern "C" int cml_forests_sample_stats(cml_forests* f, uint64_t* scratch_bytes, uint64_t* chunks, float* kernel_ms) {
  if (!f) return CML_ERR_ARG;
  if (scratch_bytes) *scratch_bytes = f->sample_scratch;
  if (chunks) *chunks = f->sample_chunks;
  if (kernel_ms) *kernel_ms = f->sample_ms;
  return CML_OK;
}

extern "C" int cml_forests_sample(cml_forests* f, const cml_forest_batch* b, uint32_t n, uint64_t seed, const uint64_t* key,
                                  double* ln_weight, uint32_t* n_and, uint64_t* base, uint32_t* nodes, uint64_t cap,
                                  double* ln_total) {
  if (!f) return CML_ERR_ARG;
  F_REQUIRE(b && ln_total && (!n || (ln_weight && n_and && base)), CML_ERR_ARG, "cml_forests_sample: null argument");
  F_REQUIRE(f->have_params, CML_ERR_STATE, "cml_forests_sample before cml_forests_set_params");
  const uint64_t nf = b->n_forests;
  F_REQUIRE(nf == 0 || (b->node_off && b->next && b->label && b->backref), CML_ERR_ARG, "cml_forests_sample: null array");
  CML_CUDA(cudaSetDevice(f->device));
  f->sample_ms = 0;
  f->sample_scratch = 0;
  f->sample_chunks = 0;
  if (n) base[0] = 0;
  if (!nf) return CML_OK;
  ForestLevels L;
  if (const int rc = forest_levelise(f, b, "cml_forests_sample", L)) return rc;
  const uint64_t n_nodes = b->node_off[nf];
  // chunk scratch: per pre-order node its inside value and largest size; per forest its total and, per sample, its
  // weight, size and output offset
  const uint64_t per_node = sizeof(double) + sizeof(uint32_t), per_forest = sizeof(double) + 20ull * n;
  const ForestChunks P = forest_chunks(b, per_node, per_forest, f->kbest_scratch_mb << 20);
  const uint64_t n_chunks = P.begin.size() - 1;
  cudaStream_t s = f->stream;
  const unsigned max_blocks = (unsigned)f->sm_count * 16u;
  const unsigned grid_cap = std::max(1u, std::min(f_cdiv(P.max_forests, kFsWarps), max_blocks));
  const uint32_t stride = std::max(1u, L.max_levels);
  const uint64_t walkers = n ? (uint64_t)grid_cap * kFsWarps * 32 : 0;
  DevArray<uint64_t> d_off, d_lvlb, d_key, d_obase;
  DevArray<uint32_t> d_next, d_label, d_order, d_lvl, d_big, d_nand, d_out;
  DevArray<uint8_t> d_br;
  DevArray<double> d_ins, d_tot, d_lnw;
  DevArray<uint2> d_stack;
  CML_CUDA(d_off.upload(b->node_off, nf + 1, s));
  CML_CUDA(d_next.upload(b->next, n_nodes, s));
  CML_CUDA(d_label.upload(b->label, n_nodes, s));
  CML_CUDA(d_br.upload(b->backref, n_nodes, s));
  CML_CUDA(d_order.upload(L.order.data(), n_nodes, s));
  CML_CUDA(d_lvl.upload(L.lvl.data(), L.lvl.size(), s));
  CML_CUDA(d_lvlb.upload(L.lvl_base.data(), nf + 1, s));
  if (key && n) CML_CUDA(d_key.upload(key, nf, s));
  CML_CUDA(d_ins.alloc(P.max_nodes));
  CML_CUDA(d_big.alloc(P.max_nodes));
  CML_CUDA(d_tot.alloc(P.max_forests));
  CML_CUDA(d_lnw.alloc(std::max<uint64_t>(1, P.max_forests * n)));
  CML_CUDA(d_nand.alloc(std::max<uint64_t>(1, P.max_forests * n)));
  CML_CUDA(d_obase.alloc(std::max<uint64_t>(1, P.max_forests * n)));
  CML_CUDA(d_stack.alloc(std::max<uint64_t>(1, walkers * stride)));
  f->sample_chunks = n_chunks;
  f->sample_scratch = P.max_nodes * per_node + P.max_forests * per_forest + walkers * stride * sizeof(uint2);
  FsArgs A{d_off.p, d_next.p, d_label.p, d_br.p, d_order.p, d_lvl.p, d_lvlb.p, f->ln_w.p, key && n ? d_key.p : nullptr,
           seed, 0, 0, 0, n, d_ins.p, d_big.p, d_stack.p, stride, d_tot.p, d_lnw.p, d_nand.p};
  EventPair ev, ev_paths;  // k_forest_sample, k_forest_sample_paths
  CML_CUDA(ev.create());
  CML_CUDA(ev_paths.create());
  bool fits = true;
  std::vector<uint64_t> obase;
  for (uint64_t c = 0; c < n_chunks; ++c) {
    const uint64_t f0 = P.begin[c], nfc = P.begin[c + 1] - f0, e0 = f0 * n, ne = nfc * n;
    A.f0 = f0;
    A.s0 = b->node_off[f0];
    A.n_f = (uint32_t)nfc;
    const unsigned grid = std::max(1u, std::min(f_cdiv(nfc, kFsWarps), grid_cap));
    CML_CUDA(cudaEventRecord(ev.a, s));
    k_forest_sample<<<grid, kFsWarps * 32, 0, s>>>(A);
    ++f->launches;
    CML_CUDA(cudaGetLastError());
    CML_CUDA(cudaEventRecord(ev.b, s));
    CML_CUDA(cudaMemcpyAsync(ln_total + f0, d_tot.p, nfc * sizeof(double), cudaMemcpyDeviceToHost, s));
    if (ne) {
      CML_CUDA(cudaMemcpyAsync(ln_weight + e0, d_lnw.p, ne * sizeof(double), cudaMemcpyDeviceToHost, s));
      CML_CUDA(cudaMemcpyAsync(n_and + e0, d_nand.p, ne * sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
    }
    CML_CUDA(cudaStreamSynchronize(s));
    float ms = 0;
    CML_CUDA(cudaEventElapsedTime(&ms, ev.a, ev.b));
    f->sample_ms += ms;
    if (!ne) continue;
    obase.resize(ne);
    for (uint64_t i = 0; i < ne; ++i) {
      F_REQUIRE(n_and[e0 + i] != kFkNone, CML_ERR_ARG,
                "cml_forests_sample: forest " + std::to_string(f0 + i / n) + " has a derivation of more than 2^32 - 2 AND nodes");
      obase[i] = base[e0 + i] - base[e0];
      base[e0 + i + 1] = base[e0 + i] + n_and[e0 + i];
    }
    const uint64_t total = base[e0 + ne] - base[e0];
    fits = fits && (!nodes || base[e0 + ne] <= cap);
    if (!nodes || !fits || !total) continue;
    if (d_out.n < total) CML_CUDA(d_out.alloc(total));
    CML_CUDA(cudaMemcpyAsync(d_obase.p, obase.data(), ne * sizeof(uint64_t), cudaMemcpyHostToDevice, s));
    CML_CUDA(cudaEventRecord(ev_paths.a, s));
    k_forest_sample_paths<<<std::min(f_cdiv(ne, kFsWarps * 32), grid_cap), kFsWarps * 32, 0, s>>>(A, d_obase.p, d_out.p);
    ++f->launches;
    CML_CUDA(cudaGetLastError());
    CML_CUDA(cudaEventRecord(ev_paths.b, s));
    CML_CUDA(cudaMemcpyAsync(nodes + base[e0], d_out.p, total * sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
    CML_CUDA(cudaStreamSynchronize(s));
    CML_CUDA(cudaEventElapsedTime(&ms, ev_paths.a, ev_paths.b));
    f->sample_ms += ms;
  }
  F_REQUIRE(!n || !nodes || base[nf * n] <= cap, CML_ERR_ARG,
            "cml_forests_sample: nodes buffer too small (need base[n_forests * n] = " + std::to_string(base[nf * n]) + ")");
  return CML_OK;
}
