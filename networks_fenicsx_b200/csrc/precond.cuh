// Network Schur-complement preconditioner (replaces PCLU/MUMPS, solver.py:58-65).
//
// The saddle-point operator of assembly.py:253-277 is condensed exactly, graph edge by graph
// edge, onto the bifurcation multipliers:
//   pressure rows   q_{a+1} - q_a = r_p[a]              =>  q_a = q_0 + F_a   (prefix sums F)
//   sum of the flux rows of an edge (pressure telescopes)
//                   W q_0 + w.F + lam_v - lam_u = sum r_q =>  q_0 = g (c + lam_u - lam_v)
//                   (w = row sums of the edge mass matrix, W = sum w = sum_j R_j h_j, g = 1/W)
//   multiplier rows => weighted graph Laplacian  L lam = rhs  with conductances g.
// On a tree network L is eliminated leaf -> root without fill; the tree is cut into chunks
// (subtrees) that one thread block solves level by level, plus one top chunk.  Graph edges that
// close a cycle ("chords") keep their conductance on the diagonal only, so P is then an SPD
// support-graph approximation and the outer FGMRES absorbs the difference.
// Back-substitution restores q by the prefix sums and p by the flux-row recurrence.
// P is built from cell_rh = R*h written by the assembly kernel, i.e. from the same element data
// as A; P^{-1} A = I up to rounding on forests.
#pragma once

#include <type_traits>

#include "assemble.cuh"
#include "peer.cuh"
#include "spmv.cuh"

namespace nxfx {

struct TreeDev {
  const int32_t* __restrict__ t_of_bif;
  const int32_t* __restrict__ bif_of_t;
  const int32_t* __restrict__ t_parent;
  const int32_t* __restrict__ t_pedge;
  const int32_t* __restrict__ t_pslot;  // flux slot of t_pedge (N == 1: cell_rh is stored in slot order)
  const int32_t* __restrict__ t_cptr;
  const int32_t* __restrict__ t_cidx;
  const int32_t* __restrict__ chunk_lptr;
  const int32_t* __restrict__ lvl_ptr;
  const int32_t* __restrict__ chunk_desc;  // [n_chunks][kDescInts]: {b0, b1, cb, ce, nl, lvl[0..nl]}
  const int32_t* __restrict__ t_inc_ptr;   // incidences of every node in SCHEDULE order (N == 1 fusion)
  const int2* __restrict__ t_inc;          // {2 * flux slot | is_in, graph edge}
  double* diag0;
  double* tg;  // conductance of the link to the parent (0 for roots)
  double* d;
  double* gd;
  double* r;
  double* lam;      // schedule order
  double* lam_nat;  // natural (bifurcation) order, read by the back-substitution
  int cap;          // chunk capacity of the shared-memory sweeps (2048 or 4096)
  // multi-GPU: the SHARED nodes of this rank's top chunk (positions inside the chunk, in the global order
  // every rank uses); the other top-chunk nodes are private to the rank and complete without exchange
  const int32_t* __restrict__ top_sh_pos;
  int n_sh;
  int sh_lmax, pr_lmin;  // deepest level of the top chunk holding a shared node / shallowest holding a private one
};

// N == 1 fusion: the tree kernels can evaluate a node's Laplacian diagonal / right-hand side on the
// fly from (r, cell_rh) while they stage a chunk, instead of reading arrays that a separate kernel
// filled (one launch and one 8-byte-per-node round trip less).  r == nullptr: not fused.
struct FusedN1 {
  Net g;
  const double* r;
  const double* cell_rh;
  const double* lam_weight = nullptr;  // multi-GPU: weight of this rank's copy of a multiplier row
};

// Development aid (-DNXFX_TREE_STAMPS): %globaltimer stamps of the phases of the fused tree kernel, taken by
// thread 0 of block 0 (slots 0..15) and of the top-chunk block (slots 16..31).
#ifdef NXFX_TREE_STAMPS
__device__ unsigned long long g_tree_stamps[32];
__device__ __forceinline__ void tree_stamp(bool top, int k) {
  if (threadIdx.x == 0 && (blockIdx.x == 0 || top)) {
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    g_tree_stamps[(top ? 16 : 0) + k] = t;
  }
}
#define NXFX_STAMP(top, k) tree_stamp((top), (k))
#else
#define NXFX_STAMP(top, k) ((void)0)
#endif

// n = node in schedule order; its incidences come from the schedule-ordered table (two dependent
// loads instead of the five of bif_of_t -> bif_ptr -> bif_inc -> edge_slot -> r).
// Per incidence (graph edge e in flux slot s, conductance g = 1 / (R h)):
//   condensed edge flux  gc = g (r_q0 + r_q1) - r_p / 2      [= ((r_q0 + r_q1) - (R h / 2) r_p) / (R h)]
//   rhs += r_p + gc (in-edge) | -gc (out-edge),   diag += g
// ONE division per incidence (FP64 divisions are ~30 dependent instructions; they were a third of the
// staging time), and the incidences are taken two at a time so that their gathers are in flight together.
// The sums run in incidence order: deterministic, identical in every kernel that stages a node.
struct IncTerm {
  double s, g;
};
__device__ __forceinline__ IncTerm n1_inc_term(const double* __restrict__ r, const double* __restrict__ cell_rh,
                                               int poff, int2 inc, double2 rq, double rp, double rh) {
  const double g = 1.0 / rh;
  const double gc = g * (rq.x + rq.y) - 0.5 * rp;
  return IncTerm{(inc.x & 1) ? (rp + gc) : -gc, g};
}

template <bool RHS, bool DIAG>
__device__ __forceinline__ void n1_node_eval(const FusedN1& f, const TreeDev& t, int n, double& s_out, double& d_out) {
  const double* __restrict__ r = f.r;
  const double* __restrict__ crh = f.cell_rh;
  const int2* __restrict__ tinc = t.t_inc;
  const int poff = f.g.poff;
  const int k0 = t.t_inc_ptr[n], k1 = t.t_inc_ptr[n + 1];
  double s = 0.0, d = 0.0;
  if (RHS) {
    const int bi = t.bif_of_t[n];
    s = f.lam_weight ? -f.lam_weight[bi] * r[f.g.loff + bi] : -r[f.g.loff + bi];
  }
  int k = k0;
  for (; k + 2 <= k1; k += 2) {
    const int2 i0 = tinc[k], i1 = tinc[k + 1];
    const double h0 = crh[i0.x >> 1], h1 = crh[i1.x >> 1];
    if (RHS) {
      const double2 q0 = *reinterpret_cast<const double2*>(r + (i0.x & ~1));
      const double2 q1 = *reinterpret_cast<const double2*>(r + (i1.x & ~1));
      const double p0 = r[poff + i0.y], p1 = r[poff + i1.y];
      const IncTerm a = n1_inc_term(r, crh, poff, i0, q0, p0, h0);
      const IncTerm b = n1_inc_term(r, crh, poff, i1, q1, p1, h1);
      s += a.s;
      s += b.s;
      if (DIAG) { d += a.g; d += b.g; }
    } else {
      d += 1.0 / h0;
      d += 1.0 / h1;
    }
  }
  if (k < k1) {
    const int2 i0 = tinc[k];
    const double h0 = crh[i0.x >> 1];
    if (RHS) {
      const double2 q0 = *reinterpret_cast<const double2*>(r + (i0.x & ~1));
      const IncTerm a = n1_inc_term(r, crh, poff, i0, q0, r[poff + i0.y], h0);
      s += a.s;
      if (DIAG) d += a.g;
    } else {
      d += 1.0 / h0;
    }
  }
  s_out = s;
  d_out = d;
}

__device__ __forceinline__ double n1_node_rhs(const FusedN1& f, const TreeDev& t, int n) {
  double s, d;
  n1_node_eval<true, false>(f, t, n, s, d);
  return s;
}

// both at once (one pass over the incidences; same operations in the same order as the two others)
__device__ __forceinline__ double n1_node_rhs_diag(const FusedN1& f, const TreeDev& t, int n, double& diag) {
  double s;
  n1_node_eval<true, true>(f, t, n, s, diag);
  return s;
}

__device__ __forceinline__ double n1_node_diag(const FusedN1& f, const TreeDev& t, int n) {
  double s, d;
  n1_node_eval<false, true>(f, t, n, s, d);
  return d;
}

// (Measured and rejected, round 2: a prefetch.global.L2 pass over all of a chunk's gather addresses before the
// evaluation -- the staging is bound by DRAM throughput on scattered 32-byte sectors, not by the latency of the
// dependent loads -- and ordering a node's incidences by graph edge instead of by flux slot: r_p gathers get
// contiguous, R h / r_q gathers lose what they gain; 48.5 vs 50.6 sectors per warp and incidence.)
#ifndef NXFX_TREE_PAIR
#define NXFX_TREE_PAIR 1
#endif

// schedule-ordered incidence table (built once per schedule)
__global__ void __launch_bounds__(kThreads)
t_inc_len_kernel(int n_bif, const int32_t* __restrict__ bif_of_t, const int32_t* __restrict__ bif_ptr,
                 int32_t* __restrict__ len) {
  const int n = blockIdx.x * blockDim.x + threadIdx.x;
  if (n > n_bif) return;
  len[n] = n < n_bif ? bif_ptr[bif_of_t[n] + 1] - bif_ptr[bif_of_t[n]] : 0;
}
__global__ void __launch_bounds__(kThreads)
t_inc_fill_kernel(int n_bif, const int32_t* __restrict__ bif_of_t, const int32_t* __restrict__ bif_ptr,
                  const int32_t* __restrict__ bif_inc, const int32_t* __restrict__ edge_slot,
                  const int32_t* __restrict__ t_inc_ptr, int2* __restrict__ t_inc) {
  const int n = blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= n_bif) return;
  const int bi = bif_of_t[n];
  int o = t_inc_ptr[n];
  const int k0 = bif_ptr[bi], deg = bif_ptr[bi + 1] - k0;
  for (int k = k0; k < k0 + deg; ++k, ++o) {
    const int inc = bif_inc[k], e = inc >> 1;
    t_inc[o] = make_int2(2 * edge_slot[e] | (inc & 1), e);
  }
}

// R h of the cells of edge e start at cell_rh + rh_base(g, e): the one-cell-per-edge assembly stores them in flux-slot
// order (assemble.cuh), otherwise they are in cell order.  (The N == 1 kernels below index by slot themselves; the
// general kernels also run with N == 1 when the schedule does not fit the shared-memory sweeps.)
__device__ __forceinline__ size_t rh_base(const Net& g, int e) {
  return g.N == 1 ? (size_t)g.edge_slot[e] : (size_t)e * g.N;
}

// g_e = 1 / sum_j R_j h_j
__global__ void __launch_bounds__(kThreads)
edge_conductance_kernel(Net g, const double* __restrict__ cell_rh, double* __restrict__ edge_g) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= g.E) return;
  const double* rh = cell_rh + rh_base(g, e);
  double W = 0.0;
  for (int j = 0; j < g.N; ++j) W += rh[j];
  edge_g[e] = 1.0 / W;
}

__global__ void __launch_bounds__(kThreads)
bif_diag_kernel(Net g, TreeDev t, const double* __restrict__ edge_g) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= g.n_bif) return;
  double s = 0.0;
  for (int k = g.bif_ptr[i]; k < g.bif_ptr[i + 1]; ++k) s += edge_g[g.bif_inc[k] >> 1];
  const int n = t.t_of_bif[i];
  t.diag0[n] = s;
  const int pe = t.t_pedge[n];
  t.tg[n] = pe >= 0 ? edge_g[pe] : 0.0;
}

// ---- shared-memory tree sweeps ------------------------------------------------------------------
// One thread block per bottom chunk: the chunk's node data, child lists and level table are staged
// in shared memory once, the level loop then runs on-chip.  Per-level latency is what bounds these
// kernels, so (i) the factorisation stores 1/d (no division on the dependent chain of the solve),
// (ii) levels with <= 32 nodes at the shallow end of a chunk are handled by ONE warp with
// __syncwarp instead of a block barrier, (iii) blocks are small (256 threads).
// The block that finishes last (atomic ticket) eliminates the top chunk.  For the solve, all blocks
// are co-resident (cooperative launch): they wait on an epoch flag for the top chunk and then
// back-substitute their chunk straight from shared memory -- one launch per preconditioner
// application.  Trees with more chunks than resident blocks use two launches (up, down).
// Chunk capacity is a launch-time parameter (TreeDev::cap): 2048 nodes per chunk keeps two blocks
// resident per SM (single-launch cooperative solve up to ~20 generations of a binary tree); 4096
// is selected by the schedule builder when the top chunk would not fit otherwise (24-25
// generations, > 100 M DOFs).  Child links: 2 * cap (the top chunk also lists its bottom-chunk children).
constexpr int kChunkCapMax = 4096;
constexpr int kLevelCap = 64;  // levels per chunk held in shared memory
constexpr int kDescInts = 8 + kLevelCap + 1;  // {b0, b1, cb, ce, nl, Lw, -, -, lvl[0..nl]}
#ifndef NXFX_TREE_THREADS
#define NXFX_TREE_THREADS 1024
#endif
constexpr int kTreeThreads = NXFX_TREE_THREADS;

struct TreeSmem {  // view of the dynamic shared memory of a tree kernel
  double* a;  // F: d -> 1/d   solve: r -> lam      [cap]
  double* b;  // F: tg         solve: 1/d           [cap]
  double* c;  // F: gd         solve: gd            [cap]
  int* cptr;  // [cap + 4]
  int* cidx;  // [2 cap]
  int* par;   // [cap]
  int* lvl;   // [kLevelCap + 3]
  int* last;
};
// behind `last`: uint32 shbits[cap / 32] -- top chunk of a partitioned network: bit i = node i is SHARED
// (replicated, exchanged), else private to this rank.  A bit array, not bytes: two resident blocks must stay
// below the 196 KB shared-memory carve-out (2 KB more per block pushed the SM to the next carve-out, halved
// its L1 and cost the staging gathers 10 us).  Not a member of the view: the single-GPU kernels run at the
// 32-register limit and must not carry a pointer they never use.
__device__ __forceinline__ unsigned int* tree_shbits(const TreeSmem& S) {
  return reinterpret_cast<unsigned int*>(S.last + 1);
}
__device__ __forceinline__ bool tree_shared(const TreeSmem& S, int i) {
  return (tree_shbits(S)[i >> 5] >> (i & 31)) & 1u;
}

__host__ __device__ constexpr size_t tree_smem_bytes(int cap) {
  return (size_t)cap * (3 * sizeof(double) + 4 * sizeof(int)) + (size_t)(4 + kLevelCap + 3 + 1) * sizeof(int) + (size_t)cap / 8;
}

__device__ __forceinline__ TreeSmem tree_view(unsigned char* raw, int cap) {
  TreeSmem S;
  S.a = reinterpret_cast<double*>(raw);
  S.b = S.a + cap;
  S.c = S.b + cap;
  S.cptr = reinterpret_cast<int*>(S.c + cap);
  S.cidx = S.cptr + cap + 4;
  S.par = S.cidx + 2 * cap;
  S.lvl = S.par + cap;
  S.last = S.lvl + kLevelCap + 3;
  return S;
}

enum { kTreeFactor = 0, kTreeUp = 1, kTreeDown = 2, kTreeUpDown = 3 };  // kTreeUpDown: a top chunk, forward then backward

struct ChunkInfo {
  int b0, b1, cb, ce, nl, Lw;  // Lw: levels 0..Lw all have <= 32 nodes (warp phase), -1 if none
};

__device__ __forceinline__ ChunkInfo load_chunk_info(const TreeDev& t, int chunk, const TreeSmem& S) {
  const int32_t* __restrict__ desc = t.chunk_desc + (size_t)chunk * kDescInts;
  ChunkInfo ci{desc[0], desc[1], desc[2], desc[3], desc[4], desc[5]};
  for (int i = threadIdx.x; i <= ci.nl; i += blockDim.x) S.lvl[i] = desc[8 + i];
  return ci;
}

// leaf -> root over the chunk's levels: block phase for the wide levels, one warp for the narrow top
// `which` (top chunk of a partitioned network): the heavy nodes private to this rank are eliminated first
// (kPrivateNodes), the shared ones after their partial sums have been exchanged (kSharedNodes).
enum { kPrivateNodes = 1, kSharedNodes = 2 };

template <typename NodeOp>
__device__ __forceinline__ void sweep_up(const TreeSmem& S, const ChunkInfo& ci, NodeOp op) {
  const int tid = threadIdx.x;
  for (int L = ci.nl - 1; L > ci.Lw; --L) {
    for (int n = S.lvl[L] + tid; n < S.lvl[L + 1]; n += blockDim.x) op(n);
    __syncthreads();
  }
  if (tid < 32) {
    for (int L = min(ci.Lw, ci.nl - 1); L >= 0; --L) {
      for (int n = S.lvl[L] + tid; n < S.lvl[L + 1]; n += 32) op(n);
      __syncwarp();
    }
  }
  __syncthreads();
}

// Partitioned network, top chunk: only the private (which = kPrivateNodes) or only the shared nodes, and only
// the levels [Llo, Lhi] that hold such nodes (the private nodes sit in the deep levels of the top chunk, the
// shared ones in the shallow levels: a level without selected nodes would still cost its barrier).
template <typename NodeOp>
__device__ __forceinline__ void sweep_up_sel(const TreeSmem& S, const ChunkInfo& ci, NodeOp op, int which, int Llo, int Lhi) {
  const int tid = threadIdx.x;
  Lhi = min(Lhi, ci.nl - 1);
  auto take = [&](int n) { return tree_shared(S, n - ci.b0) == (which == kSharedNodes); };
  for (int L = Lhi; L > ci.Lw && L >= Llo; --L) {
    for (int n = S.lvl[L] + tid; n < S.lvl[L + 1]; n += blockDim.x)
      if (take(n)) op(n);
    __syncthreads();
  }
  if (tid < 32) {
    for (int L = min(ci.Lw, Lhi); L >= Llo; --L) {
      for (int n = S.lvl[L] + tid; n < S.lvl[L + 1]; n += 32)
        if (take(n)) op(n);
      __syncwarp();
    }
  }
  __syncthreads();
}

// top chunk: flags of the shared nodes (all zero on a single GPU)
__device__ __forceinline__ void load_shared_flags(const TreeDev& t, const ChunkInfo& ci, const TreeSmem& S) {
  unsigned int* bits = tree_shbits(S);
  for (int w = threadIdx.x; w < t.cap / 32; w += blockDim.x) bits[w] = 0u;
  __syncthreads();
  for (int k = threadIdx.x; k < t.n_sh; k += blockDim.x) atomicOr(bits + (t.top_sh_pos[k] >> 5), 1u << (t.top_sh_pos[k] & 31));
  __syncthreads();
}

// root -> leaf
template <typename NodeOp>
__device__ __forceinline__ void sweep_down(const TreeSmem& S, const ChunkInfo& ci, NodeOp op) {
  const int tid = threadIdx.x;
  if (tid < 32) {
    for (int L = 0; L <= min(ci.Lw, ci.nl - 1); ++L) {
      for (int n = S.lvl[L] + tid; n < S.lvl[L + 1]; n += 32) op(n);
      __syncwarp();
    }
  }
  __syncthreads();
  for (int L = ci.Lw + 1; L < ci.nl; ++L) {
    for (int n = S.lvl[L] + tid; n < S.lvl[L + 1]; n += blockDim.x) op(n);
    __syncthreads();
  }
}

// The same two sweeps over a chunk whose data stay in global memory (tree_sweep_kernel, btree_top_split_kernel):
// the chunk's levels [L0, L1) straight from the schedule, every level strided over the whole block and closed by a
// block barrier.
template <typename NodeOp>
__device__ __forceinline__ void levels_up(const TreeDev& t, int L0, int L1, NodeOp op) {
  for (int L = L1 - 1; L >= L0; --L) {
    const int b = t.lvl_ptr[L], e = t.lvl_ptr[L + 1];
    for (int n = b + threadIdx.x; n < e; n += blockDim.x) op(n);
    __syncthreads();
  }
}

template <typename NodeOp>
__device__ __forceinline__ void levels_down(const TreeDev& t, int L0, int L1, NodeOp op) {
  for (int L = L0; L < L1; ++L) {
    const int b = t.lvl_ptr[L], e = t.lvl_ptr[L + 1];
    for (int n = b + threadIdx.x; n < e; n += blockDim.x) op(n);
    __syncthreads();
  }
}

__device__ __forceinline__ void load_children(const TreeDev& t, const ChunkInfo& ci, const TreeSmem& S) {
  const int nn = ci.b1 - ci.b0;
  for (int i = threadIdx.x; i <= nn; i += blockDim.x) S.cptr[i] = t.t_cptr[ci.b0 + i] - ci.cb;
  for (int i = threadIdx.x; i < ci.ce - ci.cb; i += blockDim.x) S.cidx[i] = t.t_cidx[ci.cb + i];
}

// Phases of the top chunk of a partitioned network around a host-driven all-reduce (tree_top_split_kernel).
enum { kPartial = 1, kFinish = 2 };

// stage a chunk for the solve: a = r, b = 1/d, c = gd, par
__device__ __forceinline__ void load_solve_chunk(const TreeDev& t, const TreeSmem& S, int b0, int b1,
                                                 const FusedN1* f = nullptr) {
  const int nn = b1 - b0;
  for (int i = threadIdx.x; i < nn; i += blockDim.x) {
    S.a[i] = f ? n1_node_rhs(*f, t, b0 + i) : t.r[b0 + i];
    S.b[i] = t.d[b0 + i];
    S.c[i] = t.gd[b0 + i];
    S.par[i] = t.t_parent[b0 + i];
  }
}

// ---- node operations ------------------------------------------------------------------------------
// What a leaf -> root sweep computes at a node, over the TreeSmem view of a staged chunk:
//   FactorOp       d_n = diag0_n - sum_c tg_c gd_c; 1/d_n, gd_n = tg_n / d_n    a: d -> 1/d   b: tg        c: gd
//   SolveOp        r_n += sum_c gd_c r_c                                     a: r          b: 1/d       c: gd
//   FactorSolveOp  both in one pass                                         a: r          b: d -> 1/d  c: gd   e: tg
// Each one provides
//   stage(f)                 the chunk's own values (all threads of the block; f: from (r, R h), N == 1)
//   fold_bottom(i)           children below b0 -- roots of bottom chunks, in global memory (top chunk)
//   eliminate<CH, PIVOT>(n)  node n from its children that pass the filter CH, then (PIVOT) the pivot;
//                            without the pivot it only folds the children in (partitioned top chunk)
//   field(q, j)              exchanged partial sum q of shared node j, in the order of the exchange buffer
//   park / restore           the global scratch that carries the top chunk from kPartial to kFinish
//   store(i)                 the results of node i to global memory
// The filter is spelled out in every child loop: behind a helper function the compiler schedules the
// single-GPU sweeps differently.
enum { kAllChildren = 0, kSharedChildren = 1, kPrivateChildren = 2 };

struct FactorOp {
  const TreeDev& t;
  const TreeSmem& S;
  int b0, b1;
  static constexpr int kFields = 2;  // [partial d | tg]
  static constexpr bool kSolves = false;

  __device__ __forceinline__ void stage(const FusedN1* f) const {
    const int nn = b1 - b0, tid = threadIdx.x, nth = blockDim.x;
    for (int i = tid; i < nn; i += nth) S.par[i] = t.t_parent[b0 + i];
    if (f) {
      for (int i = tid; i < nn; i += nth) {
        S.a[i] = n1_node_diag(*f, t, b0 + i);
        const int pe = t.t_pslot[b0 + i];
        const double tg = pe >= 0 ? 1.0 / f->cell_rh[pe] : 0.0;
        S.b[i] = tg;
        // the top chunk reads the link conductances of its bottom-chunk children (the chunk roots)
        const int p = t.t_parent[b0 + i];
        if (p < b0 || p >= b1) t.tg[b0 + i] = tg;
      }
    } else {
      for (int i = tid; i < nn; i += nth) { S.a[i] = t.diag0[b0 + i]; S.b[i] = t.tg[b0 + i]; }
    }
  }
  __device__ __forceinline__ void fold_bottom(int i) const {
    double acc = S.a[i];
    for (int k = S.cptr[i]; k < S.cptr[i + 1]; ++k) {
      const int c = S.cidx[k];
      if (c < b0) acc -= t.tg[c] * __ldcg(t.gd + c);
    }
    S.a[i] = acc;
  }
  template <int CH, bool PIVOT = true>
  __device__ __forceinline__ void eliminate(int n) const {
    const int i = n - b0;
    double acc = S.a[i];
    for (int k = S.cptr[i]; k < S.cptr[i + 1]; ++k) {
      const int c = S.cidx[k] - b0;
      if (c >= 0 && (CH == kAllChildren || tree_shared(S, c) == (CH == kSharedChildren))) acc -= S.b[c] * S.c[c];
    }
    if (!PIVOT) {
      S.a[i] = acc;
      return;
    }
    const double inv = 1.0 / acc;
    S.a[i] = inv;
    S.c[i] = S.b[i] * inv;
  }
  __device__ __forceinline__ double& field(int q, int j) const { return q == 0 ? S.a[j] : S.b[j]; }
  // private nodes: final (1/d, gd); shared nodes: (partial d, tg)
  __device__ __forceinline__ void park(int i) const {
    t.d[b0 + i] = S.a[i];
    t.gd[b0 + i] = tree_shared(S, i) ? S.b[i] : S.c[i];
  }
  __device__ __forceinline__ void restore(int i) const { S.a[i] = t.d[b0 + i]; S.c[i] = t.gd[b0 + i]; S.b[i] = 0.0; }
  __device__ __forceinline__ void store(int i) const { t.d[b0 + i] = S.a[i]; t.gd[b0 + i] = S.c[i]; }
};

struct SolveOp {
  const TreeDev& t;
  const TreeSmem& S;
  int b0, b1;
  static constexpr int kFields = 1;  // [partial rhs]
  static constexpr bool kSolves = true;

  __device__ __forceinline__ void stage(const FusedN1* f) const { load_solve_chunk(t, S, b0, b1, f); }
  __device__ __forceinline__ void fold_bottom(int i) const {
    double acc = S.a[i];
    for (int k = S.cptr[i]; k < S.cptr[i + 1]; ++k) {
      const int c = S.cidx[k];
      if (c < b0) acc += t.gd[c] * __ldcg(t.r + c);
    }
    S.a[i] = acc;
  }
  template <int CH, bool PIVOT = true>  // (a solve has no pivot)
  __device__ __forceinline__ void eliminate(int n) const {
    const int i = n - b0;
    double acc = S.a[i];
    for (int k = S.cptr[i]; k < S.cptr[i + 1]; ++k) {
      const int c = S.cidx[k] - b0;
      if (c >= 0 && (CH == kAllChildren || tree_shared(S, c) == (CH == kSharedChildren))) acc += S.c[c] * S.a[c];
    }
    S.a[i] = acc;
  }
  __device__ __forceinline__ double& field(int, int j) const { return S.a[j]; }
  __device__ __forceinline__ void park(int i) const { t.lam[b0 + i] = S.a[i]; }
  __device__ __forceinline__ void restore(int i) const {
    S.a[i] = t.lam[b0 + i];
    S.b[i] = t.d[b0 + i];
    S.c[i] = t.gd[b0 + i];
    S.par[i] = t.t_parent[b0 + i];
  }
  __device__ __forceinline__ void store(int i) const { t.r[b0 + i] = S.a[i]; }
};

// Factorisation fused with the first solve (N == 1): the leaf -> root sweep of the factorisation and the forward
// elimination of the first right-hand side visit the same nodes in the same order, so they share one staging pass
// and one set of level barriers.  A fourth shared array e = tg sits behind the TreeSmem view (the parent needs
// tg_c and gd_c of its children).
__host__ __device__ constexpr size_t tree_smem_bytes_fs(int cap) {
  return ((tree_smem_bytes(cap) + 15) & ~(size_t)15) + (size_t)cap * sizeof(double);
}
__device__ __forceinline__ double* tree_smem_e(unsigned char* raw, int cap) {
  return reinterpret_cast<double*>(raw + ((tree_smem_bytes(cap) + 15) & ~(size_t)15));
}

struct FactorSolveOp {
  const TreeDev& t;
  const TreeSmem& S;
  int b0, b1;
  // behind the view; factor_solve_up passes its own __restrict__ copy (without it the compiler schedules the
  // single-GPU sweeps differently)
  double* Se = tree_smem_e(reinterpret_cast<unsigned char*>(S.a), t.cap);
  static constexpr int kFields = 3;  // [partial d | tg | partial rhs]
  static constexpr bool kSolves = true;

  __device__ __forceinline__ void stage(const FusedN1& f) const {
    const int nn = b1 - b0, tid = threadIdx.x, nth = blockDim.x;
    if (f.cell_rh) {  // one cell per edge: diagonals / right-hand sides straight from (r, R h)
      for (int i = tid; i < nn; i += nth) {
        double dg;
        S.a[i] = n1_node_rhs_diag(f, t, b0 + i, dg);
        S.b[i] = dg;
        const int pe = t.t_pslot[b0 + i];
        const double tg = pe >= 0 ? 1.0 / f.cell_rh[pe] : 0.0;
        Se[i] = tg;
        const int p = t.t_parent[b0 + i];
        S.par[i] = p;
        if (p < b0 || p >= b1) t.tg[b0 + i] = tg;  // chunk roots: read by the top chunk
      }
    } else {  // several cells per edge: the node arrays were filled by bif_diag_kernel / bif_rhs_kernel
      for (int i = tid; i < nn; i += nth) {
        S.a[i] = t.r[b0 + i];
        S.b[i] = t.diag0[b0 + i];
        Se[i] = t.tg[b0 + i];
        S.par[i] = t.t_parent[b0 + i];
      }
    }
  }
  __device__ __forceinline__ void fold_bottom(int i) const {
    double ad = S.b[i], ar = S.a[i];
    for (int k = S.cptr[i]; k < S.cptr[i + 1]; ++k) {
      const int c = S.cidx[k];
      if (c < b0) {
        const double gdc = __ldcg(t.gd + c);
        ad -= __ldcg(t.tg + c) * gdc;
        ar += gdc * __ldcg(t.r + c);
      }
    }
    S.b[i] = ad;
    S.a[i] = ar;
  }
  template <int CH, bool PIVOT = true>
  __device__ __forceinline__ void eliminate(int n) const {
    const int i = n - b0;
    double ad = S.b[i], ar = S.a[i];
    int k = S.cptr[i];
    const int k1 = S.cptr[i + 1];
#if NXFX_TREE_PAIR
    // binary nodes: the loads of both children are issued together (the level's cost is its dependent chain);
    // the sums run in the same order as the loop below
    for (; k + 2 <= k1; k += 2) {
      const int c0 = S.cidx[k] - b0, c1 = S.cidx[k + 1] - b0;
      const int j0 = max(c0, 0), j1 = max(c1, 0);
      const double e0 = Se[j0], g0 = S.c[j0], a0 = S.a[j0];
      const double e1 = Se[j1], g1 = S.c[j1], a1 = S.a[j1];
      if (c0 >= 0 && (CH == kAllChildren || tree_shared(S, c0) == (CH == kSharedChildren))) { ad -= e0 * g0; ar += g0 * a0; }
      if (c1 >= 0 && (CH == kAllChildren || tree_shared(S, c1) == (CH == kSharedChildren))) { ad -= e1 * g1; ar += g1 * a1; }
    }
#endif
    for (; k < k1; ++k) {
      const int c = S.cidx[k] - b0;
      if (c >= 0 && (CH == kAllChildren || tree_shared(S, c) == (CH == kSharedChildren))) {
        ad -= Se[c] * S.c[c];
        ar += S.c[c] * S.a[c];
      }
    }
    if (!PIVOT) {
      S.b[i] = ad;
      S.a[i] = ar;
      return;
    }
    const double inv = 1.0 / ad;
    S.b[i] = inv;
    S.c[i] = Se[i] * inv;
    S.a[i] = ar;
  }
  __device__ __forceinline__ double& field(int q, int j) const { return q == 0 ? S.b[j] : (q == 1 ? Se[j] : S.a[j]); }
  // private nodes: final (1/d, gd) and eliminated rhs; shared nodes: (partial d, tg) and partial rhs
  __device__ __forceinline__ void park(int i) const {
    t.d[b0 + i] = S.b[i];
    t.gd[b0 + i] = tree_shared(S, i) ? Se[i] : S.c[i];
    t.lam[b0 + i] = S.a[i];
  }
  __device__ __forceinline__ void restore(int i) const {
    S.b[i] = t.d[b0 + i];
    S.c[i] = t.gd[b0 + i];
    S.a[i] = t.lam[b0 + i];
    Se[i] = 0.0;
    S.par[i] = t.t_parent[b0 + i];
  }
  __device__ __forceinline__ void store(int i) const { t.d[b0 + i] = S.b[i]; t.gd[b0 + i] = S.c[i]; }
};

// ---- top chunk of a partitioned network ----------------------------------------------------------
// The top chunk holds nodes PRIVATE to this rank, which complete locally, and SHARED ones, which every rank
// holds (t.top_sh_pos).  (1) eliminate the private nodes; (2) fold them into their shared parents; (3) the caller
// sums the partial sums of the shared nodes (Op::field) over the ranks, in rank order; (4) eliminate the shared
// nodes from their shared children -- identically on every rank.  A private node has no shared child.
template <typename Op>
__device__ __forceinline__ void top_partial(const Op& op, const ChunkInfo& ci) {
  const TreeDev& t = op.t;
  sweep_up_sel(op.S, ci, [&](int n) { op.template eliminate<kAllChildren>(n); }, kPrivateNodes, t.pr_lmin, 1 << 30);
  for (int k = threadIdx.x, nth = blockDim.x; k < t.n_sh; k += nth)
    op.template eliminate<kPrivateChildren, false>(ci.b0 + t.top_sh_pos[k]);
  __syncthreads();
}

template <typename Op>
__device__ __forceinline__ void top_finish(const Op& op, const ChunkInfo& ci) {
  sweep_up_sel(op.S, ci, [&](int n) { op.template eliminate<kSharedChildren>(n); }, kSharedNodes, 0, op.t.sh_lmax);
}

// numeric factorisation of one chunk; t.d receives 1/d.  `top`: children below b0 live in bottom chunks (already
// written to HBM).
__device__ __forceinline__ void factor_chunk(const TreeDev& t, const TreeSmem& S, int chunk, bool top, const FusedN1* f) {
  const ChunkInfo ci = load_chunk_info(t, chunk, S);
  const FactorOp op{t, S, ci.b0, ci.b1};
  const int nn = ci.b1 - ci.b0, tid = threadIdx.x, nth = blockDim.x;
  load_children(t, ci, S);
  op.stage(f);
  __syncthreads();
  if (top) {
    for (int i = tid; i < nn; i += nth) op.fold_bottom(i);
    __syncthreads();
  }
  sweep_up(S, ci, [&](int n) { op.eliminate<kAllChildren>(n); });
  for (int i = tid; i < nn; i += nth) op.store(i);
}

// load a chunk for the solve: child lists and load_solve_chunk
__device__ __forceinline__ ChunkInfo stage_solve_chunk(const TreeDev& t, const TreeSmem& S, int chunk,
                                                       const FusedN1* f = nullptr) {
  const ChunkInfo ci = load_chunk_info(t, chunk, S);
  load_children(t, ci, S);
  load_solve_chunk(t, S, ci.b0, ci.b1, f);
  __syncthreads();
  return ci;
}

// forward elimination of a staged chunk: r_n += sum_c gd_c r_c
__device__ __forceinline__ void solve_up(const TreeDev& t, const TreeSmem& S, const ChunkInfo& ci, bool top) {
  const SolveOp op{t, S, ci.b0, ci.b1};
  const int nn = ci.b1 - ci.b0, tid = threadIdx.x, nth = blockDim.x;
  if (top) {
    for (int i = tid; i < nn; i += nth) op.fold_bottom(i);
    __syncthreads();
  }
  sweep_up(S, ci, [&](int n) { op.eliminate<kAllChildren>(n); });
  for (int i = tid; i < nn; i += nth) op.store(i);
}

// lam = r/d + gd * lam(parent); parents outside the chunk (top chunk) are read through L2
// `top`: only the top chunk's multipliers are read by other chunks (through t.lam, schedule order)
__device__ __forceinline__ void solve_down(const TreeDev& t, const TreeSmem& S, const ChunkInfo& ci, bool top) {
  const int b0 = ci.b0, b1 = ci.b1, nn = ci.b1 - ci.b0;
  sweep_down(S, ci, [&](int n) {
    const int i = n - b0;
    const int p = S.par[i];
    double v = S.a[i] * S.b[i];
    if (p >= b0 && p < b1) v += S.c[i] * S.a[p - b0];
    else if (p >= 0) v += S.c[i] * __ldcg(t.lam + p);
    S.a[i] = v;
  });
  for (int i = threadIdx.x; i < nn; i += blockDim.x) {
    if (top) t.lam[b0 + i] = S.a[i];
    t.lam_nat[t.bif_of_t[b0 + i]] = S.a[i];
  }
}

// true in the block that finished last
__device__ __forceinline__ bool last_block_done(const TreeSmem& S, unsigned int* ticket, int n_bottom) {
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) *S.last = (atomicAdd(ticket, 1u) == (unsigned int)n_bottom - 1);
  __syncthreads();
  const bool last = *S.last != 0;
  if (last) __threadfence();
  return last;
}

// grid = max(n_bottom, 1); do_top = 0 (multi-GPU): bottom chunks only
__global__ void __launch_bounds__(kTreeThreads)
tree_factor_kernel(TreeDev t, int n_bottom, unsigned int* ticket, int do_top, FusedN1 fin) {
  extern __shared__ __align__(16) unsigned char tree_smem_raw[];
  TreeSmem S = tree_view(tree_smem_raw, t.cap);
  const FusedN1* f = fin.cell_rh ? &fin : nullptr;
  if (n_bottom > 0) {
    factor_chunk(t, S, blockIdx.x, false, f);
    if (!do_top) return;
    if (!last_block_done(S, ticket, n_bottom)) return;
  }
  if (!do_top) return;
  factor_chunk(t, S, n_bottom, true, f);
  if (threadIdx.x == 0) *ticket = 0u;
}

// MODE kTreeUp: forward sweep of the bottom chunks, top chunk (forward + backward) in the last
// block.  MODE kTreeDown: backward sweep of the bottom chunks.  (two-launch path)
template <int MODE>
__global__ void __launch_bounds__(kTreeThreads)
tree_solve_kernel(TreeDev t, int n_bottom, unsigned int* ticket, int do_top) {
  extern __shared__ __align__(16) unsigned char tree_smem_raw[];
  TreeSmem S = tree_view(tree_smem_raw, t.cap);
  if (MODE == kTreeDown) {
    const ChunkInfo ci = stage_solve_chunk(t, S, blockIdx.x);
    solve_down(t, S, ci, false);
    return;
  }
  if (n_bottom > 0) {
    const ChunkInfo ci = stage_solve_chunk(t, S, blockIdx.x);
    solve_up(t, S, ci, false);
    for (int i = threadIdx.x; i < ci.b1 - ci.b0; i += blockDim.x) t.r[ci.b0 + i] = S.a[i];
    if (!do_top) return;
    if (!last_block_done(S, ticket, n_bottom)) return;
  }
  if (!do_top) return;
  const ChunkInfo ti = stage_solve_chunk(t, S, n_bottom);
  solve_up(t, S, ti, true);
  solve_down(t, S, ti, true);
  if (threadIdx.x == 0) *ticket = 0u;
}

// single-launch solve: grid = n_bottom + 1 co-resident blocks (cooperative launch; two blocks per
// SM, <= 32 registers, so that 20 generations fit 148 SMs).  The last block owns the top chunk: it
// stages it while the bottom blocks sweep, waits for their roots (ticket), solves the top chunk and
// raises the epoch flag; the bottom blocks then back-substitute straight from shared memory.
__global__ void __launch_bounds__(kTreeThreads, 2)
tree_solve_coop_kernel(TreeDev t, int n_bottom, unsigned int* ticket, unsigned int* flag, unsigned int epoch,
                       FusedN1 fin) {
  extern __shared__ __align__(16) unsigned char tree_smem_raw[];
  TreeSmem S = tree_view(tree_smem_raw, t.cap);
  const FusedN1* f = fin.r ? &fin : nullptr;
  const ChunkInfo ci = stage_solve_chunk(t, S, blockIdx.x, f);
  if ((int)blockIdx.x == n_bottom) {
    if (threadIdx.x == 0) {
      while (atomicAdd(ticket, 0u) != (unsigned int)n_bottom) __nanosleep(32);
      __threadfence();
    }
    __syncthreads();
    solve_up(t, S, ci, true);
    solve_down(t, S, ci, true);
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) {
      *ticket = 0u;
      __threadfence();
      atomicExch(flag, epoch);
    }
    return;
  }
  solve_up(t, S, ci, false);
  for (int i = threadIdx.x; i < ci.b1 - ci.b0; i += blockDim.x)
    if (S.par[i] < ci.b0 || S.par[i] >= ci.b1) t.r[ci.b0 + i] = S.a[i];
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) {
    atomicAdd(ticket, 1u);
    while (atomicAdd(flag, 0u) != epoch) __nanosleep(64);
    __threadfence();
  }
  __syncthreads();
  solve_down(t, S, ci, false);
}

// Factorisation + first forward elimination of one chunk (FactorSolveOp).
// wait_ticket (top chunk in its own block): the chunk's own values are staged first, then the block
// waits until all wait_count bottom blocks have published their roots.
// pc (top chunk, multi-GPU): the partial sums of the shared nodes are exchanged with the other ranks over NVLink
// inside the kernel, between top_partial and top_finish.
template <bool DIST = false>
__device__ __forceinline__ void factor_solve_up(const TreeDev& t, const TreeSmem& S, double* __restrict__ Se,
                                                const ChunkInfo& ci, bool top, const FusedN1& f,
                                                unsigned int* wait_ticket = nullptr, int wait_count = 0,
                                                const PeerDev* pc = nullptr) {
  const FactorSolveOp op{t, S, ci.b0, ci.b1, Se};
  const int nn = ci.b1 - ci.b0, tid = threadIdx.x, nth = blockDim.x;
  op.stage(f);
  __syncthreads();
  NXFX_STAMP(top, 3);
  if (top) {  // fold in the bottom-chunk children (written by the other blocks of this launch)
    if (wait_ticket) {
      if (tid == 0) {
        while (atomicAdd(wait_ticket, 0u) != (unsigned int)wait_count) __nanosleep(32);
        __threadfence();
      }
      __syncthreads();
    }
    NXFX_STAMP(top, 4);
    for (int i = tid; i < nn; i += nth) op.fold_bottom(i);
    __syncthreads();
    NXFX_STAMP(top, 5);
  }
  if (DIST && top && pc && pc->nranks > 1 && t.n_sh > 0) {
    const int ns = t.n_sh;
    const int32_t* __restrict__ pos = t.top_sh_pos;
    load_shared_flags(t, ci, S);
    top_partial(op, ci);
    NXFX_STAMP(top, 12);
    peer_ll_send(*pc, 0, FactorSolveOp::kFields * ns, [&](int i) { return op.field(i / ns, pos[i % ns]); });
    __syncthreads();  // the partial sums have been read out of shared memory: they may be overwritten
    for (int k = tid; k < ns; k += nth) {
      double v[FactorSolveOp::kFields] = {};
      for (int src = 0; src < pc->nranks; ++src)  // rank order: the same sums on every rank
#pragma unroll
        for (int q = 0; q < FactorSolveOp::kFields; ++q) v[q] += peer_ll_recv(*pc, 0, src, q * ns + k);
#pragma unroll
      for (int q = 0; q < FactorSolveOp::kFields; ++q) op.field(q, pos[k]) = v[q];
    }
    __syncthreads();
    NXFX_STAMP(top, 13);
    top_finish(op, ci);
  } else {
    // single GPU / bottom chunks: the plain level sweep (the latency-critical loop carries nothing else)
    sweep_up(S, ci, [&](int n) { op.eliminate<kAllChildren>(n); });
  }
  NXFX_STAMP(top, 6);
  for (int i = tid; i < nn; i += nth) op.store(i);
  NXFX_STAMP(top, 7);
}

// grid = n_bottom + 1 co-resident blocks (cooperative launch).  The LAST block owns the top chunk: it
// stages the chunk's own diagonals / right-hand sides while the bottom blocks work, waits for their
// roots (ticket), factorises + solves the top chunk and raises the epoch flag; the bottom blocks
// then back-substitute their chunk straight from shared memory.
// MULTI: more bottom chunks than co-resident blocks.  Bottom block k then takes the chunks k, k + G, k + 2G, ...
// (G = bottom blocks in the grid): every chunk but its last is written back in full (eliminated right-hand
// sides next to the factors) and re-staged for the backward sweep; the last one stays in shared memory.
template <bool DIST, bool MULTI>
__global__ void __launch_bounds__(kTreeThreads, 2)
tree_factor_solve_coop_kernel(TreeDev t, int n_bottom, unsigned int* ticket, unsigned int* flag, unsigned int epoch,
                              FusedN1 fin, PeerDev pc) {
  extern __shared__ __align__(16) unsigned char tree_smem_raw[];
  TreeSmem S = tree_view(tree_smem_raw, t.cap);
  double* Se = tree_smem_e(tree_smem_raw, t.cap);
  const int G = (int)gridDim.x - 1;  // bottom blocks; the last block of the grid owns the top chunk
  const bool is_top = (int)blockIdx.x == G;
  NXFX_STAMP(is_top, 0);
  const ChunkInfo ci = load_chunk_info(t, is_top ? n_bottom : (int)blockIdx.x, S);
  load_children(t, ci, S);
  NXFX_STAMP(is_top, 1);
  // programmatic dependent launch: the schedule tables above are static; everything below reads the
  // output of the preceding kernels.  Dependents (the back-substitution) are released only now, so
  // that whatever they read before their own wait is complete as well.
  asm volatile("griddepcontrol.wait;" ::: "memory");
  asm volatile("griddepcontrol.launch_dependents;");
  NXFX_STAMP(is_top, 2);
  if (is_top) {
    factor_solve_up<DIST>(t, S, Se, ci, true, fin, ticket, n_bottom, &pc);
    solve_down(t, S, ci, true);
    NXFX_STAMP(true, 10);
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) {
      *ticket = 0u;
      __threadfence();
      atomicExch(flag, epoch);
    }
    NXFX_STAMP(true, 11);
    return;
  }
  if (DIST) fin.lam_weight = nullptr;  // only shared multipliers (top chunk) carry a weight other than 1
  if (!MULTI) {  // one chunk per block: it stays in shared memory from the first load to the last store
    factor_solve_up(t, S, Se, ci, false, fin);
    // publish the eliminated right-hand sides of the chunk roots for the top chunk
    for (int i = threadIdx.x; i < ci.b1 - ci.b0; i += blockDim.x)
      if (S.par[i] < ci.b0 || S.par[i] >= ci.b1) t.r[ci.b0 + i] = S.a[i];
    __threadfence();
    __syncthreads();
    NXFX_STAMP(false, 8);
    if (threadIdx.x == 0) {
      atomicAdd(ticket, 1u);
      while (atomicAdd(flag, 0u) != epoch) __nanosleep(64);
      __threadfence();
    }
    __syncthreads();
    NXFX_STAMP(false, 9);
    solve_down(t, S, ci, false);
    NXFX_STAMP(false, 10);
    return;
  }
  int chunk = (int)blockIdx.x;
  ChunkInfo cm = ci;
  while (true) {
    const bool more = chunk + G < n_bottom;
    factor_solve_up(t, S, Se, cm, false, fin);
    // the chunk roots for the top chunk -- and every node of a chunk that has to leave shared memory
    for (int i = threadIdx.x; i < cm.b1 - cm.b0; i += blockDim.x)
      if (more || S.par[i] < cm.b0 || S.par[i] >= cm.b1) t.r[cm.b0 + i] = S.a[i];
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) atomicAdd(ticket, 1u);
    if (!more) break;
    chunk += G;
    cm = load_chunk_info(t, chunk, S);
    load_children(t, cm, S);
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    while (atomicAdd(flag, 0u) != epoch) __nanosleep(64);
    __threadfence();
  }
  __syncthreads();
  solve_down(t, S, cm, false);
  for (int c = (int)blockIdx.x; c < chunk; c += G) {  // the chunks that were written back
    __syncthreads();
    const ChunkInfo cj = load_chunk_info(t, c, S);
    load_solve_chunk(t, S, cj.b0, cj.b1);
    __syncthreads();
    solve_down(t, S, cj, false);
  }
}

// Multi-GPU form of the fused factor + first solve: bottom chunks only (no top chunk, no backward
// sweep); the top chunk follows in tree_top_split_kernel<FactorSolveOp, *>.
__global__ void __launch_bounds__(kTreeThreads, 2)
tree_factor_solve_bottom_kernel(TreeDev t, FusedN1 fin) {
  extern __shared__ __align__(16) unsigned char tree_smem_raw[];
  TreeSmem S = tree_view(tree_smem_raw, t.cap);
  double* Se = tree_smem_e(tree_smem_raw, t.cap);
  const ChunkInfo ci = load_chunk_info(t, blockIdx.x, S);
  load_children(t, ci, S);
  factor_solve_up(t, S, Se, ci, false, fin);
  for (int i = threadIdx.x; i < ci.b1 - ci.b0; i += blockDim.x) t.r[ci.b0 + i] = S.a[i];
}

// Top chunk of a partitioned network alone (one block), in two phases around the caller's SUM all-reduce of
// buf = Op::kFields x n_sh doubles, the exchanged partial sums of the shared nodes.  kPartial folds in this rank's
// bottom-chunk children, runs steps 1 and 2, parks every node in global scratch and packs buf; kFinish restores
// the scratch, takes the shared nodes from the reduced buf, runs step 4 and, for a solve, the backward sweep.
// fin: the fused input of FactorSolveOp, which stages the chunk as the single-GPU top chunk does (it also fills
// par and the link conductances t.tg of the roots).  The host-driven FactorOp / SolveOp split stages from the
// node arrays and does not read fin.  FactorSolveOp::stage takes fin by reference while the other two take a
// pointer: taking the address of a kernel parameter copies it to local memory, and the single-GPU kernels keep
// the form they had.
template <typename Op, int PHASE>
__global__ void __launch_bounds__(kTreeThreads)
tree_top_split_kernel(TreeDev t, int top_chunk, double* buf, FusedN1 fin) {
  extern __shared__ __align__(16) unsigned char tree_smem_raw[];
  TreeSmem S = tree_view(tree_smem_raw, t.cap);
  const ChunkInfo ci = load_chunk_info(t, top_chunk, S);
  const Op op{t, S, ci.b0, ci.b1};
  const int nn = ci.b1 - ci.b0, ns = t.n_sh, tid = threadIdx.x, nth = blockDim.x;
  const int32_t* __restrict__ pos = t.top_sh_pos;
  load_children(t, ci, S);
  load_shared_flags(t, ci, S);
  if (PHASE == kPartial) {
    if constexpr (std::is_same<Op, FactorSolveOp>::value) op.stage(fin);  // from (r, R h)
    else op.stage(nullptr);                                                 // from the node arrays
    __syncthreads();
    for (int i = tid; i < nn; i += nth) op.fold_bottom(i);
    __syncthreads();
    top_partial(op, ci);
    for (int i = tid; i < nn; i += nth) op.park(i);
    for (int k = tid; k < ns; k += nth)
#pragma unroll
      for (int q = 0; q < Op::kFields; ++q) buf[q * ns + k] = op.field(q, pos[k]);
  } else {
    for (int i = tid; i < nn; i += nth) op.restore(i);
    __syncthreads();
    for (int k = tid; k < ns; k += nth)
#pragma unroll
      for (int q = 0; q < Op::kFields; ++q) op.field(q, pos[k]) = buf[q * ns + k];
    __syncthreads();
    top_finish(op, ci);
    // every node, as after a whole-chunk sweep: a private node writes back the final values kPartial parked
    for (int i = tid; i < nn; i += nth) op.store(i);
    if (Op::kSolves) solve_down(t, S, ci, true);
  }
}

// ---- global-memory sweeps -----------------------------------------------------------------------------
// For schedules that do not fit the shared-memory kernels, and for the 2 x 2 blocks of the higher-order
// condensation (condense.cuh BlockFactor / BlockSolve).  A node op reads and writes global memory and provides
//   own(n)        the node's own value
//   fold(v, c)    child c folded into v
//   store(n, v)   the node's results from its folded value (a factorisation pivots here)
// and a solve op also down(n), the node of the backward sweep.
// ScalarFactor: d_n = diag0_n - sum_c g_c gd_c ;  t.d <- 1/d_n ;  gd_n = g_n / d_n
struct ScalarFactor {
  const TreeDev& t;
  const double* __restrict__ edge_g;
  __device__ __forceinline__ double own(int n) const { return t.diag0[n]; }
  __device__ __forceinline__ void fold(double& d, int c) const { d -= edge_g[t.t_pedge[c]] * t.gd[c]; }
  __device__ __forceinline__ void store(int n, double d) const {
    t.d[n] = 1.0 / d;  // the solve multiplies by 1/d
    const int pe = t.t_pedge[n];
    t.gd[n] = pe >= 0 ? edge_g[pe] / d : 0.0;
  }
};

// ScalarSolve: forward r_n += sum_c gd_c r_c ;  backward lam_n = r_n / d_n + gd_n lam_parent
struct ScalarSolve {
  const TreeDev& t;
  __device__ __forceinline__ double own(int n) const { return t.r[n]; }
  __device__ __forceinline__ void fold(double& r, int c) const { r += t.gd[c] * t.r[c]; }
  __device__ __forceinline__ void store(int n, double r) const { t.r[n] = r; }
  __device__ __forceinline__ void down(int n) const {
    const int p = t.t_parent[n];
    double v = t.r[n] * t.d[n];
    if (p >= 0) v += t.gd[n] * t.lam[p];
    t.lam[n] = v;
    t.lam_nat[t.bif_of_t[n]] = v;
  }
};

// node n of a whole-chunk sweep: its children in t_cidx order
template <typename Op>
__device__ __forceinline__ void eliminate_node(const TreeDev& t, const Op& op, int n) {
  const int c0 = t.t_cptr[n], c1 = t.t_cptr[n + 1];
  auto v = op.own(n);
  for (int k = c0; k < c1; ++k) op.fold(v, t.t_cidx[k]);
  op.store(n, v);
}

// MODE kTreeFactor / kTreeUp (leaf -> root), kTreeDown (root -> leaf), kTreeUpDown (top chunk) over one chunk.
template <int MODE, typename Factor, typename Solve>
__device__ __forceinline__ void sweep_chunk(const TreeDev& t, int chunk, const Factor& factor, const Solve& solve) {
  const int L0 = t.chunk_lptr[chunk], L1 = t.chunk_lptr[chunk + 1];
  if (MODE == kTreeFactor) levels_up(t, L0, L1, [&](int n) { eliminate_node(t, factor, n); });
  if (MODE == kTreeUp || MODE == kTreeUpDown) levels_up(t, L0, L1, [&](int n) { eliminate_node(t, solve, n); });
  if (MODE == kTreeDown || MODE == kTreeUpDown) levels_down(t, L0, L1, [&](int n) { solve.down(n); });
}

// One thread block per chunk; chunk = blockIdx.x + chunk0.  The block form, btree_sweep_kernel (condense.cuh), is a
// kernel of its own: edge_g is read through the read-only cache only as a __restrict__ kernel parameter.
template <int MODE>
__global__ void __launch_bounds__(1024)
tree_sweep_kernel(TreeDev t, const double* __restrict__ edge_g, int chunk0) {
  sweep_chunk<MODE>(t, chunk0 + blockIdx.x, ScalarFactor{t, edge_g}, ScalarSolve{t});
}

// Edge condensation: c_e = sum r_q - w.F,  F_N = sum r_p
// WITH_G (fresh matrix + direct solve): also the conductance g_e = 1 / sum_j R_j h_j of edge_conductance_kernel,
// from the same pass over R h (same sum, same order)
template <bool WITH_G = false>
__global__ void __launch_bounds__(kThreads)
edge_condense_kernel(Net g, const double* __restrict__ cell_rh, const double* __restrict__ r,
                     double* __restrict__ edge_c, double* __restrict__ edge_fn, double* __restrict__ edge_g = nullptr) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= g.E) return;
  const int N = g.N;
  const double* rq = r + (size_t)g.edge_slot[e] * (N + 1);
  const double* rp = r + g.poff + (size_t)e * N;
  const double* rh = cell_rh + rh_base(g, e);
  double s = 0.0, F = 0.0, wF = 0.0, hl = 0.0, W = 0.0;
  for (int a = 0; a <= N; ++a) {
    s += rq[a];
    const double hr = a < N ? rh[a] : 0.0;
    if (WITH_G) W += hr;
    wF += 0.5 * (hl + hr) * F;
    if (a < N) F += rp[a];
    hl = hr;
  }
  edge_c[e] = s - wF;
  edge_fn[e] = F;
  if (WITH_G) edge_g[e] = 1.0 / W;
}

// rhs_b = -r_lam + sum_in (F_N + g c) - sum_out g c      (schedule order)
// lam_weight (multi-GPU): 0 on the ranks that hold a replicated multiplier without owning it, so
// that -r_lambda is counted once in the all-reduced right-hand side; null = all ones.
// WITH_DIAG (fresh matrix + direct solve): also the Laplacian diagonal and the link conductance of
// bif_diag_kernel, from the same pass over the incidences
template <bool WITH_DIAG = false>
__global__ void __launch_bounds__(kThreads)
bif_rhs_kernel(Net g, TreeDev t, const double* __restrict__ r, const double* __restrict__ edge_g,
               const double* __restrict__ edge_c, const double* __restrict__ edge_fn,
               const double* __restrict__ lam_weight) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= g.n_bif) return;
  double s = lam_weight ? -lam_weight[i] * r[g.loff + i] : -r[g.loff + i];
  double d = 0.0;
  for (int k = g.bif_ptr[i]; k < g.bif_ptr[i + 1]; ++k) {
    const int inc = g.bif_inc[k], e = inc >> 1;
    const double ge = edge_g[e];
    const double gc = ge * edge_c[e];
    s += (inc & 1) ? (edge_fn[e] + gc) : -gc;
    if (WITH_DIAG) d += ge;
  }
  const int n = t.t_of_bif[i];
  t.r[n] = s;
  if (WITH_DIAG) {
    t.diag0[n] = d;
    const int pe = t.t_pedge[n];
    t.tg[n] = pe >= 0 ? edge_g[pe] : 0.0;
  }
}

// Back-substitution: q_a = q_0 + F_a ; p_0 = r_q0 + lam_u - (Mq)_0 ; p_a = p_{a-1} + r_qa - (Mq)_a
// ADD: z += P^{-1} r (iterative refinement updates x in place).
template <bool ADD>
__global__ void __launch_bounds__(kThreads)
edge_backsub_kernel(Net g, TreeDev t, const double* __restrict__ cell_rh,
                    const double* __restrict__ r, const double* __restrict__ edge_g,
                    const double* __restrict__ edge_c, double* __restrict__ z) {
  // let a dependent residual kernel (launched with programmatic stream serialisation) move in and
  // prefetch its first matrix tiles while this grid drains
  asm volatile("griddepcontrol.launch_dependents;");
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= g.E) {
    const int i = idx - g.E;
    if (i < g.n_bif) { if (ADD) z[g.loff + i] += t.lam_nat[i]; else z[g.loff + i] = t.lam_nat[i]; }
    return;
  }
  const int e = idx, N = g.N;
  const int slot = g.edge_slot[e];
  const int4 uv = g.slot_uvl[slot];
  const double lu = uv.z >= 0 ? t.lam_nat[uv.z] : 0.0;
  const double lv = uv.w >= 0 ? t.lam_nat[uv.w] : 0.0;
  const double* rq = r + (size_t)slot * (N + 1);
  const double* rp = r + g.poff + (size_t)e * N;
  const double* rh = cell_rh + rh_base(g, e);
  double* zq = z + (size_t)slot * (N + 1);
  double* zp = z + g.poff + (size_t)e * N;
  const double q0 = edge_g[e] * (edge_c[e] + lu - lv);
  double F = 0.0, qprev = 0.0, qa = q0, hl = 0.0, p = lu;
  for (int a = 0; a <= N; ++a) {
    if (ADD) zq[a] += qa; else zq[a] = qa;
    double qn = 0.0, hr = 0.0;
    if (a < N) {
      F += rp[a];
      qn = q0 + F;
      hr = rh[a];
      const double Mq = hl * (qprev * kSixth + qa * kThird) + hr * (qa * kThird + qn * kSixth);
      p += rq[a] - Mq;
      if (ADD) zp[a] += p; else zp[a] = p;
    }
    qprev = qa;
    qa = qn;
    hl = hr;
  }
}

// ---- N == 1 specialisations -------------------------------------------------------------------------
// With one cell per edge the condensation is  c = r_q0 + r_q1 - (rh/2) r_p,  F_N = r_p,  g = 1/rh:
// cheap enough to recompute where it is needed, so the per-edge arrays (edge_g, edge_c, edge_fn)
// and the kernels that fill them disappear from the N == 1 path.
__global__ void __launch_bounds__(kThreads)
bif_diag_n1_kernel(Net g, TreeDev t, const double* __restrict__ cell_rh) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= g.n_bif) return;
  double s = 0.0;
  for (int k = g.bif_ptr[i]; k < g.bif_ptr[i + 1]; ++k) s += 1.0 / cell_rh[g.edge_slot[g.bif_inc[k] >> 1]];
  const int n = t.t_of_bif[i];
  t.diag0[n] = s;
  const int pe = t.t_pslot[n];
  t.tg[n] = pe >= 0 ? 1.0 / cell_rh[pe] : 0.0;
}

__global__ void __launch_bounds__(kThreads)
bif_rhs_n1_kernel(Net g, TreeDev t, const double* __restrict__ r, const double* __restrict__ cell_rh,
                  const double* __restrict__ lam_weight) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= g.n_bif) return;
  double s = lam_weight ? -lam_weight[i] * r[g.loff + i] : -r[g.loff + i];
  for (int k = g.bif_ptr[i]; k < g.bif_ptr[i + 1]; ++k) {
    const int inc = g.bif_inc[k], e = inc >> 1;
    const int slot = g.edge_slot[e];
    const double2 rq = *reinterpret_cast<const double2*>(r + 2 * (size_t)slot);
    const double rp = r[g.poff + e], rh = cell_rh[slot];
    const double gc = (1.0 / rh) * (rq.x + rq.y) - 0.5 * rp;  // as n1_inc_term
    s += (inc & 1) ? (rp + gc) : -gc;
  }
  t.r[t.t_of_bif[i]] = s;
}

template <bool ADD>
__global__ void __launch_bounds__(kThreads)
edge_backsub_n1_kernel(Net g, TreeDev t, const double* __restrict__ cell_rh, const double* __restrict__ r,
                       double* __restrict__ z) {
  // let a dependent residual kernel (launched with programmatic stream serialisation) move in and
  // prefetch its first matrix tiles while this grid drains
  asm volatile("griddepcontrol.launch_dependents;");
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= g.E) {
    asm volatile("griddepcontrol.wait;" ::: "memory");
    const int i = idx - g.E;
    if (i < g.n_bif) { if (ADD) z[g.loff + i] += t.lam_nat[i]; else z[g.loff + i] = t.lam_nat[i]; }
    return;
  }
  // as a programmatic dependent of the tree kernel: r and cell_rh are older than that kernel
  // (it releases its dependents only after its own wait), the multipliers are its output.
  // Thread <-> flux SLOT: the multiplier pair, the flux pair of r / z and cell_rh are contiguous accesses;
  // only the pressure entry (cell order) is indexed through slot_edge.
  const int slot = idx;
  const int2 lm = g.slot_lm[slot];
  const int e = g.slot_edge[slot];
  const double2 rq = *reinterpret_cast<const double2*>(r + 2 * (size_t)slot);
  const double rp = r[g.poff + e], rh = cell_rh[slot];
  asm volatile("griddepcontrol.wait;" ::: "memory");
  const double lu = lm.x >= 0 ? t.lam_nat[lm.x] : 0.0;
  const double lv = lm.y >= 0 ? t.lam_nat[lm.y] : 0.0;
  const double c = (rq.x + rq.y) - 0.5 * rh * rp;
  const double q0 = (c + lu - lv) / rh;
  const double q1 = q0 + rp;
  const double p = lu + rq.x - rh * (q0 * kThird + q1 * kSixth);
  double2* zq = reinterpret_cast<double2*>(z + 2 * (size_t)slot);
  if (ADD) {
    const double2 o = *zq;
    *zq = make_double2(o.x + q0, o.y + q1);
    z[g.poff + e] += p;
  } else {
    *zq = make_double2(q0, q1);
    z[g.poff + e] = p;
  }
}

// ---- multi-GPU helpers --------------------------------------------------------------------------
// shared (replicated) multiplier rows of a vector -> contiguous buffer for the all-reduce
__global__ void __launch_bounds__(kThreads)
pack_shared_kernel(int n_shared, int loff, const int32_t* __restrict__ shared_lm,
                   const double* __restrict__ v, double* __restrict__ buf) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n_shared) buf[i] = v[loff + shared_lm[i]];
}

// After the all-reduce of [shared rows of r | partial ||r||^2 | ||b||^2]: write the reduced shared
// rows back into r and finish the norms (identical on every rank).  One block.
__global__ void __launch_bounds__(kThreads)
residual_finish_kernel(int n_shared, int loff, const int32_t* __restrict__ shared_lm,
                       const double* __restrict__ buf, double* __restrict__ r, double* __restrict__ nrm_out) {
  __shared__ double red[kThreads / 32];
  double acc = 0.0;
  for (int i = threadIdx.x; i < n_shared; i += blockDim.x) {
    const double v = buf[i];
    r[loff + shared_lm[i]] = v;
    acc += v * v;
  }
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    double s = buf[n_shared];
    for (int w = 0; w < kThreads / 32; ++w) s += red[w];
    nrm_out[0] = s;
    nrm_out[1] = buf[n_shared + 1];
  }
}

// z = D^{-1} r on flux rows (D = diag of the mass block), identity elsewhere
__global__ void __launch_bounds__(kThreads)
jacobi_flux_kernel(int n, int nq, const int32_t* __restrict__ rowptr,
                   const int32_t* __restrict__ colidx, const double* __restrict__ vals,
                   const double* __restrict__ r, double* __restrict__ z) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  double v = r[i];
  if (i < nq) {
    for (int k = rowptr[i]; k < rowptr[i + 1]; ++k)
      if (colidx[k] == i) v /= vals[k];
  }
  z[i] = v;
}

}  // namespace nxfx
