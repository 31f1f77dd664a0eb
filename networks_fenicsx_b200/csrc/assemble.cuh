// Mesh generation, symbolic pattern and numeric assembly kernels.
//
// Design (DESIGN.md "Assembly"): the assembly is ROW-OWNED.  One thread owns one matrix row,
// evaluates the (at most two) element tensors that touch it from the vertex coordinates, and
// stages the row's entries in shared memory at its offset inside the block's CSR tile; the block
// then streams the tile to HBM with fully coalesced stores.  No atomics, every stored value is
// written exactly once, and a value that has two cell contributions (the mass-matrix diagonal at a
// vertex shared by two cells of one graph edge) is the IEEE sum of two operands, so the result is
// bit-reproducible and independent of any scheduling (SURVEY A.5).
//
// Forms restated here: assembly.py:253-255 (mass, +-grad . tangent), :258-262 (right-hand side),
// :271-277 (multiplier coupling); explicit zeros of the multiplier blocks as stored by DOLFINx.
// All arithmetic uses the _rn intrinsics so that ptxas cannot contract a*b+c into an FMA: the
// values are bit-identical to the NumPy oracle.
#pragma once

#include "ctx.cuh"

namespace nxfx {

// Division by a runtime constant d >= 2 without the ~25-instruction integer divide
// (libdivide's branch-free u32 scheme): q = (((n - t) >> 1) + t) >> shift, t = umulhi(n, magic).
struct FastDiv {
  uint32_t magic, shift;
};
inline FastDiv make_fastdiv(uint32_t d) {
  FastDiv f;
  uint32_t fl = 31;
  while (!((d >> fl) & 1u)) --fl;
  if ((d & (d - 1)) == 0) {
    f.magic = 0;
    f.shift = fl == 0 ? 0 : fl - 1;  // d == 1 is never passed by the kernels
  } else {
    const uint64_t n = 1ull << (32 + fl);
    uint64_t m = n / d;
    const uint64_t rem = n % d;
    m += m;
    if (2 * rem >= d) m += 1;
    f.magic = (uint32_t)(m + 1);
    f.shift = fl;
  }
  return f;
}
__device__ __forceinline__ int fastdiv(int n, FastDiv f) {
  const uint32_t t = __umulhi((uint32_t)n, f.magic);
  return (int)(((((uint32_t)n - t) >> 1) + t) >> f.shift);
}

struct Net {
  int32_t n_nodes, E, N, n_bif;
  int32_t nq, poff, loff, ndofs;
  FastDiv div_np1, div_n;  // divide by N+1 / N (valid when N >= 2)
  const int4* __restrict__ slot_uvl;
  const int2* __restrict__ slot_lm;  // [E] {lm(u), lm(v)} in slot order (N == 1 back-substitution: 8 instead of 16 bytes)
  const int32_t* __restrict__ slot_edge;
  const int32_t* __restrict__ edge_slot;
  const int32_t* __restrict__ bif_ptr;
  const int32_t* __restrict__ bif_inc;
  const double2* __restrict__ x2;  // [nv] vertex records {x, y | z, p_bc or tagged multiplier index} (32 B each)
  const int2* __restrict__ slot_uv;          // [E] {u, v} in slot order (N == 1 assembly: 8 instead of 16 bytes per edge)
  const uint32_t* __restrict__ bif_in_bits;  // bit k = incidence k is an in-edge (multiplier rows: 1 bit instead of 4 bytes)
};

// The 4th double of a vertex record holds the boundary pressure -- only ever read at BOUNDARY vertices
// (assembly.py:258-260) -- so at bifurcation vertices it carries the node's multiplier index instead, as
// a tagged NaN: the one-cell-per-edge assembly then finds lm(u), lm(v) in the records it loads anyway.
constexpr unsigned int kLmTag = 0x7FF8B1F0u;
__device__ __forceinline__ double lm_box(int lm) {
  return __hiloint2double((int)kLmTag, lm);
}
__device__ __forceinline__ int lm_unbox(double p) {  // multiplier index, or -1 at a boundary / interior vertex
  return (unsigned int)__double2hiint(p) == kLmTag ? __double2loint(p) : -1;
}

struct Coef {
  const double* __restrict__ R_cell;  // [nc] or null
  const double* __restrict__ f_cell;  // [nc] or null
  double R_const, f_const;
  double* __restrict__ cell_rh;  // [nc] out: R*h per cell, written with the matrix (lhs); N == 1: indexed by flux SLOT
};

constexpr double kThird = 1.0 / 3.0;
constexpr double kSixth = 1.0 / 6.0;
constexpr int kMaxFluxRow = 7;  // 3 mass + 2 pressure + 2 multiplier entries (flux degree 1)

__device__ __forceinline__ int vertex_id(const Net& g, int e, int u, int v, int a) {
  // mesh.py:276,292: graph nodes first, then N-1 interior points per edge in edge order
  return a == 0 ? u : (a == g.N ? v : g.n_nodes + e * (g.N - 1) + (a - 1));
}

struct VertexRec {
  double x, y, z, p;
};

// one 32-byte sector per vertex: coordinates and the boundary pressure travel together
__device__ __forceinline__ VertexRec load_vertex(const double2* __restrict__ x2, int v) {
  const double2* p = x2 + 2 * (size_t)v;
  const double2 a = __ldg(p), b = __ldg(p + 1);
  return VertexRec{a.x, a.y, b.x, b.y};
}

__device__ __forceinline__ double seg_length(const VertexRec& v0, const VertexRec& v1) {
  const double dx = __dsub_rn(v1.x, v0.x), dy = __dsub_rn(v1.y, v0.y), dz = __dsub_rn(v1.z, v0.z);
  return __dsqrt_rn(
      __dadd_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)), __dmul_rn(dz, dz)));
}

// ---- vertices ------------------------------------------------------------------------------
// mesh.py:275,290: interior point k (1..N-1) of edge (u,v) = start*(1-w) + end*w, w = k*(1/N)
__global__ void __launch_bounds__(kThreads)
pad_nodes_kernel(int n_nodes, int gdim, const double* __restrict__ pos, double* __restrict__ x) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_nodes * 3) return;
  int node = i / 3, d = i - node * 3;
  x[4 * (size_t)node + d] = d < gdim ? pos[(size_t)node * gdim + d] : 0.0;
}

// p_bc interpolated into P1 (assembly.py:225-234) is stored in the 4th slot of the vertex records
__global__ void __launch_bounds__(kThreads)
set_pbc_kernel(int64_t nv, const double* __restrict__ pbc, double* __restrict__ x) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i < nv && lm_unbox(x[4 * i + 3]) < 0) x[4 * i + 3] = pbc[i];  // bifurcation records keep their tag
}

__global__ void __launch_bounds__(kThreads)
tag_lm_kernel(int n_nodes, const int32_t* __restrict__ node_lm, double* __restrict__ x) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n_nodes && node_lm[i] >= 0) x[4 * (size_t)i + 3] = lm_box(node_lm[i]);
}

__global__ void __launch_bounds__(kThreads)
interior_vertices_kernel(int n_nodes, int E, int N, const int32_t* __restrict__ eu,
                         const int32_t* __restrict__ ev, double* __restrict__ x) {
  const int64_t total = (int64_t)E * (N - 1) * 3;
  const double step = 1.0 / (double)N;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total;
       i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t vert = i / 3;
    const int d = (int)(i - vert * 3);
    const int e = (int)(vert / (N - 1));
    const int k = (int)(vert - (int64_t)e * (N - 1)) + 1;
    const double w = __dmul_rn((double)k, step);
    const double s = x[4 * (size_t)eu[e] + d], t = x[4 * (size_t)ev[e] + d];
    x[4 * ((size_t)n_nodes + vert) + d] = __dadd_rn(__dmul_rn(s, __dsub_rn(1.0, w)), __dmul_rn(t, w));
  }
}

// ---- row decode ----------------------------------------------------------------------------
// Flux row `r` (edge slot, local vertex a): entries in ascending column order
//   [mass a-1, a, a+1] [pressure cells a-1, a] [multipliers of u and/or v]
// Column decode (symbolic phase); the numeric kernel below emits values in the same order.
__device__ __forceinline__ int flux_row_cols(const Net& g, int r, int* cols) {
  const int N = g.N, np1 = N + 1;
  const int slot = r / np1, a = r - slot * np1;
  const int4 t = g.slot_uvl[slot];
  const int e = g.slot_edge[slot];
  int n = 0;
  if (a > 0) cols[n++] = r - 1;
  cols[n++] = r;
  if (a < N) cols[n++] = r + 1;
  const int pb = g.poff + e * N;
  if (a > 0) cols[n++] = pb + a - 1;
  if (a < N) cols[n++] = pb + a;
  const bool hu = t.z >= 0 && a <= 1, hv = t.w >= 0 && a >= N - 1;
  if (hu && hv) {
    cols[n++] = g.loff + min(t.z, t.w);
    cols[n++] = g.loff + max(t.z, t.w);
  } else if (hu) {
    cols[n++] = g.loff + t.z;
  } else if (hv) {
    cols[n++] = g.loff + t.w;
  }
  return n;
}

__device__ __forceinline__ int flux_row_len(const Net& g, int r) {
  const int N = g.N, np1 = N + 1;
  const int slot = r / np1, a = r - slot * np1;
  const int4 t = g.slot_uvl[slot];
  const int inner = (a > 0) + (a < N);
  return 1 + 2 * inner + (t.z >= 0 && a <= 1) + (t.w >= 0 && a >= N - 1);
}

// ---- symbolic ------------------------------------------------------------------------------
__global__ void __launch_bounds__(kThreads) row_len_kernel(Net g, int32_t* __restrict__ len) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r > g.ndofs) return;
  int n = 0;
  if (r < g.nq) n = flux_row_len(g, r);
  else if (r < g.loff) n = 2;
  else if (r < g.ndofs) n = 2 * (g.bif_ptr[r - g.loff + 1] - g.bif_ptr[r - g.loff]);
  len[r] = n;  // len[ndofs] = 0 so that the exclusive scan yields rowptr[ndofs] = nnz
}

__global__ void __launch_bounds__(kThreads)
fill_cols_kernel(Net g, const int32_t* __restrict__ rowptr, int32_t* __restrict__ colidx) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= g.ndofs) return;
  int32_t* out = colidx + rowptr[r];
  const int np1 = g.N + 1;
  if (r < g.nq) {
    int cols[kMaxFluxRow];
    const int n = flux_row_cols(g, r, cols);
    for (int i = 0; i < n; ++i) out[i] = cols[i];
  } else if (r < g.loff) {
    const int cell = r - g.poff, e = cell / g.N, j = cell - e * g.N;
    const int fb = g.edge_slot[e] * np1;
    out[0] = fb + j;
    out[1] = fb + j + 1;
  } else {
    const int i0 = g.bif_ptr[r - g.loff], i1 = g.bif_ptr[r - g.loff + 1];
    for (int k = i0; k < i1; ++k) {
      const int inc = g.bif_inc[k], e = inc >> 1;
      const int fb = g.edge_slot[e] * np1;
      const int c0 = (inc & 1) ? fb + g.N - 1 : fb;  // in-edge: last cell; out-edge: first cell
      out[2 * (k - i0)] = c0;
      out[2 * (k - i0) + 1] = c0 + 1;
    }
  }
}

// ---- numeric -------------------------------------------------------------------------------
// One thread per matrix row.  A flux-row thread (slot, a) owns cell a of its graph edge (a < N):
// it loads the two vertex records of that cell, evaluates m_a = R_a h_a and hands m_a and the
// boundary pressure of the cell's end vertex to the next row of the same edge by warp shuffle
// (the previous cell's contribution to the shared-vertex mass entry), so every cell is evaluated
// once per warp.  Entries are staged in shared memory at the row's CSR offset (branch-free,
// predicated stores) and streamed out with 16-byte stores.  N1 = one cell per edge (compile-time
// fast path of the headline workload); otherwise N >= 2 with magic-number division.
struct SmemSink {
  double* sm;
  __device__ __forceinline__ void operator()(bool on, int idx, double v) const {
    if (on) sm[idx] = v;
  }
};
template <bool ACC>
struct GlobalSink {  // tiles larger than the staging buffer (very high degree bifurcations)
  double* vals;
  __device__ __forceinline__ void operator()(bool on, int idx, double v) const {
    if (on) {
      if (ACC) vals[idx] += v; else vals[idx] = v;
    }
  }
};

// Everything a row needs from the index tables.
struct RowDesc {
  int sbase, tnnz, start;  // tile base / size, row offset inside the tile
  int a, e;                // flux rows: local vertex, graph edge
  int4 t;                  // flux rows: {u, v, lm(u), lm(v)}
  int i0, i1;              // multiplier rows: incidence range
};

template <bool ACC, bool N1, typename Sink>
__device__ __forceinline__ void assemble_row(const Net& g, const Coef& c, const RowDesc& d, int r, int p,
                                             int lane, double* __restrict__ b, int lhs, int rhs, const Sink& put) {
  const int N = N1 ? 1 : g.N;
  // ---- flux rows: geometry phase (all lanes take part in the shuffles) ----------------------
  const bool isflux = r < g.nq;
  const int a = d.a, e = d.e;
  const int4 t = d.t;
  double mR = 0.0, pA = 0.0, pNext = 0.0;
  if (isflux) {
    if (a < N) {
      const VertexRec v0 = load_vertex(g.x2, N1 ? t.x : vertex_id(g, e, t.x, t.y, a));
      const VertexRec v1 = load_vertex(g.x2, N1 ? t.y : vertex_id(g, e, t.x, t.y, a + 1));
      const double R = c.R_cell ? c.R_cell[(size_t)e * N + a] : c.R_const;
      mR = __dmul_rn(R, seg_length(v0, v1));
      if (lhs) {  // the factorisation is built from cell_rh: it must follow the matrix (ADD_VALUES included)
        if (ACC) c.cell_rh[(size_t)e * N + a] += mR; else c.cell_rh[(size_t)e * N + a] = mR;
      }
      pA = v0.p;
      pNext = v1.p;
    }
  }
  const double mPrev = __shfl_up_sync(0xffffffffu, mR, 1);
  const double pPrev = __shfl_up_sync(0xffffffffu, pNext, 1);
  if (isflux) {
    double mL = 0.0;
    if (a > 0) {
      if (N1 || lane > 0) {  // the previous lane owns cell a-1 of the same edge
        mL = mPrev;
        if (a == N) pA = pPrev;
      } else {  // first lane of the warp: evaluate cell a-1 here
        const VertexRec v0 = load_vertex(g.x2, vertex_id(g, e, t.x, t.y, a - 1));
        const VertexRec v1 = load_vertex(g.x2, vertex_id(g, e, t.x, t.y, a));
        const double R = c.R_cell ? c.R_cell[(size_t)e * N + a - 1] : c.R_const;
        mL = __dmul_rn(R, seg_length(v0, v1));
        pA = v1.p;
      }
    }
    const bool hasL = a > 0, hasR = a < N;
    // mass block (assembly.py:253): R h [[1/3,1/6],[1/6,1/3]] per cell
    const double dL = __dmul_rn(mL, kThird), dR = __dmul_rn(mR, kThird);
    const double diag = hasL ? (hasR ? __dadd_rn(dL, dR) : dL) : dR;
    put(hasL, p, __dmul_rn(mL, kSixth));
    p += hasL;
    put(true, p, diag);
    ++p;
    put(hasR, p, __dmul_rn(mR, kSixth));
    p += hasR;
    // a[i][P] = -int p dv/ds: -B^T (assembly.py:255)
    put(hasL, p, -1.0);
    p += hasL;
    put(hasR, p, 1.0);
    p += hasR;
    // multiplier columns (assembly.py:273,277); the cell's other flux dof stores an explicit 0.0
    const bool hu = t.z >= 0 && a <= 1, hv = t.w >= 0 && a >= N - 1;
    const double vu = a == 0 ? -1.0 : 0.0, vv = a == N ? 1.0 : 0.0;
    const bool ufirst = !hv || (hu && t.z < t.w);
    put(hu || hv, p, (hu && ufirst) ? vu : vv);
    put(hu && hv, p + 1, ufirst ? vv : vu);
    if (rhs) {
      // assembly.py:258-260: +p_bc at in_marker vertices (boundary END of an edge), -p_bc at
      // out_marker vertices (boundary START of an edge)
      double bv = 0.0;
      if (a == 0 && t.z < 0) bv = -pA;
      if (a == N && t.w < 0) bv = pA;
      if (ACC) b[r] += bv; else b[r] = bv;
    }
  } else if (r < g.loff) {
    // a[P][i] = +int phi dq/ds: B = [-1, +1] (assembly.py:254);  L[P] = int f phi (assembly.py:262)
    put(true, p, -1.0);
    put(true, p + 1, 1.0);
    if (rhs) {
      double bv = 0.0;
      if (c.f_cell || c.f_const != 0.0) {
        const int cell = r - g.poff;
        const int ce = N1 ? cell : fastdiv(cell, g.div_n), j = cell - ce * N;
        const int4 ct = g.slot_uvl[g.edge_slot[ce]];
        const double h = seg_length(load_vertex(g.x2, vertex_id(g, ce, ct.x, ct.y, j)),
                                    load_vertex(g.x2, vertex_id(g, ce, ct.x, ct.y, j + 1)));
        bv = __dmul_rn(c.f_cell ? c.f_cell[cell] : c.f_const, h);
      }
      if (ACC) b[r] += bv; else b[r] = bv;
    }
  } else if (r < g.ndofs) {
    // a[LM][c] = +mu q at in-edges, -mu q at out-edges (assembly.py:272,276)
    for (int k = d.i0; k < d.i1; ++k) {
      const bool in = g.bif_inc[k] & 1;
      put(true, p, in ? 0.0 : -1.0);
      put(true, p + 1, in ? 1.0 : 0.0);
      p += 2;
    }
    if (rhs && !ACC) b[r] = 0.0;
  }
}

// ---- region-specialised tiles -----------------------------------------------------------------
// The rows of the three regions [flux | pressure | multiplier] are tiled separately, so a block
// never mixes row types:
//   flux tile      N == 1: one thread per graph EDGE emits both of its rows (no shuffles, no
//                  divergence between the a=0 / a=1 lanes), 512 rows per block;
//                  N >= 2: one thread per row with the warp-shuffle hand-over (assemble_row);
//   pressure tile  rows are the constant pair {-1, +1}: 16-byte stores straight to HBM;
//   multiplier tile the values are a function of the incidence list only: incidence-parallel.
constexpr int kFluxRowsN1 = 512;
constexpr int kAsmCap = 2560;  // 512 rows * 5 entries (N == 1)  >=  256 rows * 7 entries (N >= 2)
constexpr int kPresRows = 512;
constexpr int kLamRows = 256;

// The value / rhs streams are written once and not re-read by this kernel: streaming (evict-first)
// stores keep them from pushing the vertex records out of L2.
#define NXFX_ST2(ptr, v) __stcs((ptr), (v))
#define NXFX_ST1(ptr, v) __stcs((ptr), (v))
#define NXFX_LDS(ptr) __ldcs(ptr)
// (measured, round 2: writing the right-hand side and R*h with the default policy so that the solve finds
// them in L2 made the assembly 2 us slower and the solve no faster -- the 117 MB value stream flushes
// them anyway -- so they stream too)
#define NXFX_STB2(ptr, v) __stcs((ptr), (v))
#define NXFX_STB1(ptr, v) __stcs((ptr), (v))

template <bool ACC>
__device__ __forceinline__ void store_pair(double* __restrict__ vals, size_t idx, double v0, double v1) {
  // idx even => 16-byte aligned (vals comes from cudaMalloc)
  if ((idx & 1) == 0) {
    double2* dst = reinterpret_cast<double2*>(vals + idx);
    double2 v = make_double2(v0, v1);
    if (ACC) { const double2 o = *dst; v.x += o.x; v.y += o.y; }
    NXFX_ST2(dst, v);
  } else {
    if (ACC) { vals[idx] += v0; vals[idx + 1] += v1; } else { vals[idx] = v0; vals[idx + 1] = v1; }
  }
}

// coalesced 16-byte flush of a staged tile; entries were staged at sm[off + k], off = sbase & 1
template <bool ACC>
__device__ __forceinline__ void flush_tile(const double* sm, double* __restrict__ vals, int sbase, int tnnz) {
  const int off = sbase & 1;
  double* out = vals + sbase - off;
  const int lo = off, hi = off + tnnz;
  const int npair = (hi + 1) >> 1;
  for (int q = threadIdx.x; q < npair; q += blockDim.x) {
    const int i = 2 * q;
    if (i >= lo && i + 1 < hi) {
      double2 v = *reinterpret_cast<const double2*>(sm + i);
      double2* dst = reinterpret_cast<double2*>(out + i);
      if (ACC) { const double2 o = *dst; v.x += o.x; v.y += o.y; }
      NXFX_ST2(dst, v);
    } else {
      if (i >= lo && i < hi) { if (ACC) out[i] += sm[i]; else out[i] = sm[i]; }
      if (i + 1 >= lo && i + 1 < hi) { if (ACC) out[i + 1] += sm[i + 1]; else out[i + 1] = sm[i + 1]; }
    }
  }
}

// N == 1 flux tile: thread <-> edge slot, rows 2*slot (vertex u) and 2*slot+1 (vertex v).
// Everything the thread needs comes from its 8-byte slot record {u, v} and the two vertex records (which
// carry the multiplier index of a bifurcation vertex in place of the unused boundary pressure): the row's
// CSR offset inside the tile is 6 * (slots before) + 2 * (multiplier entries before) --
// a ballot / popcount prefix over the block instead of a strided rowptr load --, and R*h is stored in SLOT
// order (coalesced; the graph-edge index is only needed for a per-cell R array).
template <bool ACC>
__device__ __forceinline__ void flux_tile_n1(const Net& g, const Coef& c, const int32_t* __restrict__ rowptr,
                                             double* __restrict__ vals, double* __restrict__ b, int lhs,
                                             int rhs, int tile, double* sm) {
  __shared__ int warp_nl[kTileRows / 32];
  const int r0 = tile * kFluxRowsN1;
  const int slot = (r0 >> 1) + threadIdx.x;
  const bool active = slot < g.E;
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  int4 t = make_int4(0, 0, -1, -1);
  VertexRec v0, v1;
  if (active) {
    const int2 uv = NXFX_LDS(g.slot_uv + slot);
    v0 = load_vertex(g.x2, uv.x);
    v1 = load_vertex(g.x2, uv.y);
    t = make_int4(uv.x, uv.y, lm_unbox(v0.p), lm_unbox(v1.p));
  }
  const bool hu = t.z >= 0, hv = t.w >= 0;
  const unsigned bu = __ballot_sync(0xffffffffu, hu), bv = __ballot_sync(0xffffffffu, hv);
  const unsigned lt = (1u << lane) - 1u;
  int pre = __popc(bu & lt) + __popc(bv & lt);  // multiplier entry pairs of the earlier lanes
  if (lane == 0) warp_nl[w] = __popc(bu) + __popc(bv);
  const int sbase = rowptr[r0];
  double m = 0.0;
  if (active) {
    const double R = c.R_cell ? c.R_cell[NXFX_LDS(g.slot_edge + slot)] : c.R_const;
    m = __dmul_rn(R, seg_length(v0, v1));
  }
  __syncthreads();
  int tot = 0;
#pragma unroll
  for (int k = 0; k < kTileRows / 32; ++k) {
    const int v = warp_nl[k];
    if (k < w) pre += v;
    tot += v;
  }
  const int nact = min(kFluxRowsN1 >> 1, g.E - (r0 >> 1));
  const int tnnz = 6 * nact + 2 * tot;  // == rowptr[rend] - sbase
  if (active) {
    const int r = 2 * slot;
    if (rhs) {
      // assembly.py:258-260: -p_bc at out_marker vertices (boundary START), +p_bc at in_marker (END)
      const double b0 = hu ? 0.0 : -v0.p, b1 = hv ? 0.0 : v1.p;
      double2* dst = reinterpret_cast<double2*>(b + r);  // r even
      double2 v = make_double2(b0, b1);
      if (ACC) { const double2 o = *dst; v.x += o.x; v.y += o.y; }
      NXFX_STB2(dst, v);
    }
    if (lhs) {
      // the factorisation is built from cell_rh: it follows the matrix (ADD_VALUES included)
      if (ACC) c.cell_rh[slot] += m; else NXFX_STB1(c.cell_rh + slot, m);
      const double m3 = __dmul_rn(m, kThird), m6 = __dmul_rn(m, kSixth);
      const bool ufirst = !hv || (hu && t.z < t.w);
      const int nl = (int)hu + (int)hv;
      // row u: [m/3, m/6 | +1 | (lam_u: -1) (lam_v: 0)]; row v: [m/6, m/3 | -1 | (lam_u: 0) (lam_v: +1)]
      const double u0 = (hu && ufirst) ? -1.0 : 0.0, u1 = ufirst ? 0.0 : -1.0;
      const double w0 = (hu && ufirst) ? 0.0 : 1.0, w1 = ufirst ? 1.0 : 0.0;
      double* s0 = sm + (sbase & 1) + 6 * (int)threadIdx.x + 2 * pre;
      double* s1 = s0 + 3 + nl;
      s0[0] = m3; s0[1] = m6; s0[2] = 1.0;
      s1[0] = m6; s1[1] = m3; s1[2] = -1.0;
      if (nl > 0) { s0[3] = u0; s1[3] = w0; }
      if (nl > 1) { s0[4] = u1; s1[4] = w1; }
    }
  }
  if (lhs) {  // tnnz <= 256 slots * 10 entries == kAsmCap always holds for N == 1
    __syncthreads();
    flush_tile<ACC>(sm, vals, sbase, tnnz);
  }
}

// N >= 2 flux tile: thread <-> row
template <bool ACC>
__device__ __forceinline__ void flux_tile_gen(const Net& g, const Coef& c, const int32_t* __restrict__ rowptr,
                                              double* __restrict__ vals, double* __restrict__ b, int lhs,
                                              int rhs, int tile, double* sm) {
  const int r0 = tile * kTileRows;
  const int rend = min(r0 + kTileRows, g.nq);
  const int r = r0 + threadIdx.x;
  RowDesc d;
  d.sbase = rowptr[r0];
  d.tnnz = rowptr[rend] - d.sbase;
  d.start = 0; d.a = 0; d.e = 0; d.i0 = d.i1 = 0;
  d.t = make_int4(0, 0, -1, -1);
  const bool active = r < rend;
  if (active) {
    d.start = rowptr[r] - d.sbase;
    const int slot = fastdiv(r, g.div_np1);
    d.a = r - slot * (g.N + 1);
    d.t = g.slot_uvl[slot];
    d.e = g.slot_edge[slot];
  }
  const int lane = threadIdx.x & 31;
  const int rr = active ? r : g.ndofs;  // inactive lanes still take part in the shuffles
  if (d.tnnz > kAsmCap) {
    if (lhs) assemble_row<ACC, false>(g, c, d, rr, d.sbase + d.start, lane, b, lhs, rhs, GlobalSink<ACC>{vals});
    else assemble_row<ACC, false>(g, c, d, rr, 0, lane, b, lhs, rhs, [](bool, int, double) {});
    return;
  }
  assemble_row<ACC, false>(g, c, d, rr, (d.sbase & 1) + d.start, lane, b, lhs, rhs, SmemSink{sm});
  if (lhs) {
    __syncthreads();
    flush_tile<ACC>(sm, vals, d.sbase, d.tnnz);
  }
}

// pressure tile: a[P][i] = +int phi dq/ds: B = [-1, +1] (assembly.py:254); L[P] = int f phi (:262).
// lhs == 0 (rhs only, or the values are already in place: see MatState::static_valid) writes b alone.
template <bool ACC, bool N1>
__device__ __forceinline__ void pressure_tile(const Net& g, const Coef& c, const int32_t* __restrict__ rowptr,
                                              double* __restrict__ vals, double* __restrict__ b, int lhs,
                                              int rhs, int tile) {
  const int r0 = g.poff + tile * kPresRows;
  const int rend = min(r0 + kPresRows, g.loff);
  const int sbase = rowptr[r0];  // every pressure row has exactly two entries
  const int N = N1 ? 1 : g.N;
  for (int r = r0 + threadIdx.x; r < rend; r += blockDim.x) {
    if (lhs) store_pair<ACC>(vals, (size_t)sbase + 2 * (size_t)(r - r0), -1.0, 1.0);
    if (rhs) {
      double bv = 0.0;
      if (c.f_cell || c.f_const != 0.0) {
        const int cell = r - g.poff;
        const int ce = N1 ? cell : fastdiv(cell, g.div_n), j = cell - ce * N;
        const int4 ct = g.slot_uvl[g.edge_slot[ce]];
        const double h = seg_length(load_vertex(g.x2, vertex_id(g, ce, ct.x, ct.y, j)),
                                    load_vertex(g.x2, vertex_id(g, ce, ct.x, ct.y, j + 1)));
        bv = __dmul_rn(c.f_cell ? c.f_cell[cell] : c.f_const, h);
      }
      if (ACC) b[r] += bv; else NXFX_STB1(b + r, bv);
    }
  }
}

// multiplier tile: a[LM][c] = +mu q at in-edges, -mu q at out-edges (assembly.py:272,276); the
// touching cell's other flux dof stores an explicit 0.0.  Incidence k of the tile owns the pair
// at 2*(k - k0): in-edge (0, +1), out-edge (-1, 0).
template <bool ACC>
__device__ __forceinline__ void lambda_tile(const Net& g, const int32_t* __restrict__ rowptr,
                                            double* __restrict__ vals, double* __restrict__ b, int lhs,
                                            int rhs, int tile) {
  const int i0 = tile * kLamRows;
  const int i1 = min(i0 + kLamRows, g.n_bif);
  if (lhs) {
    const int k0 = g.bif_ptr[i0], k1 = g.bif_ptr[i1];
    const int sbase = rowptr[g.loff + i0];
    for (int k = k0 + threadIdx.x; k < k1; k += blockDim.x) {
      const bool in = (g.bif_in_bits[k >> 5] >> (k & 31)) & 1u;
      store_pair<ACC>(vals, (size_t)sbase + 2 * (size_t)(k - k0), in ? 0.0 : -1.0, in ? 1.0 : 0.0);
    }
  }
  if (rhs && !ACC)
    for (int i = i0 + threadIdx.x; i < i1; i += blockDim.x) NXFX_STB1(b + g.loff + i, 0.0);
}

// write_static == 0: the pressure and multiplier rows of vals already hold what this assembly would store
// there (a re-assembly without ADD_VALUES, MatState::static_valid); their tiles then write b only.
template <bool ACC, bool N1>
__global__ void __launch_bounds__(kTileRows)
assemble_tiles_kernel(Net g, Coef c, const int32_t* __restrict__ rowptr, double* __restrict__ vals,
                      double* __restrict__ b, int lhs, int rhs, int write_static, int n_flux_tiles, int n_pres_tiles) {
  __shared__ __align__(16) double sm[kAsmCap + 2];
  // a kernel launched as programmatic dependent (the fused tree kernel) may stage its schedule
  // tables while the last wave of this grid drains; it waits for this grid before reading any output
  asm volatile("griddepcontrol.launch_dependents;");
  // flux tiles first, then pressure, then multiplier tiles: each region is written as one
  // ascending stream (interleaving the tile types along the block index measured 6 % slower)
  const int t = blockIdx.x;
  if (t < n_flux_tiles) {
    if (N1) flux_tile_n1<ACC>(g, c, rowptr, vals, b, lhs, rhs, t, sm);
    else flux_tile_gen<ACC>(g, c, rowptr, vals, b, lhs, rhs, t, sm);
  } else if (t < n_flux_tiles + n_pres_tiles) {
    pressure_tile<ACC, N1>(g, c, rowptr, vals, b, lhs && write_static, rhs, t - n_flux_tiles);
  } else {
    lambda_tile<ACC>(g, rowptr, vals, b, lhs && write_static, rhs, t - n_flux_tiles - n_pres_tiles);
  }
}

// post_processing.py:36-51: per cell the two flux dofs of its edge
__global__ void __launch_bounds__(kThreads)
global_flux_kernel(Net g, const double* __restrict__ x, double* __restrict__ out) {
  const int64_t total = (int64_t)g.E * g.N;
  for (int64_t cell = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; cell < total;
       cell += (int64_t)gridDim.x * blockDim.x) {
    const int e = (int)(cell / g.N), j = (int)(cell - (int64_t)e * g.N);
    const int q0 = g.edge_slot[e] * (g.N + 1) + j;
    out[2 * cell] = x[q0];
    out[2 * cell + 1] = x[q0 + 1];
  }
}

// dst[r * N + j] = src[row(r) * S + (S == N ? j : 0)], row(r) = map ? map[r] : r, S in {1, N} (nxfx_gather)
__global__ void gather_kernel(int64_t n_rows, int N, int S, const int32_t* __restrict__ map, const double* __restrict__ src,
              double* __restrict__ dst) {
  const int64_t total = n_rows * N;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / N;
    const int j = (int)(i - r * N);
    const int64_t row = map ? (int64_t)map[r] : r;
    dst[i] = src[row * S + (S == N ? j : 0)];
  }
}

}  // namespace nxfx
