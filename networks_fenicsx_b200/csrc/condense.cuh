// Exact network condensation for general polynomial degrees (flux P_fd, pressure DG0 / continuous P_pd;
// assembly.py:121-146) -- the direct solve the reference gets from MUMPS (solver.py:58-65).
//
// Per graph edge e = (u, v) the unknowns that live on the edge only (its flux dofs, the pressure dofs inside
// it, the pressure of a boundary node at its end) are eliminated:
//     K_e y + C_e z_e = r_loc,     z_e = (P_u, lam_u, P_v, lam_v)   nodal unknowns at the bifurcations,
// K_e = banded saddle matrix (local unknowns ordered along the edge), factorised per edge by a banded LU with
// partial pivoting (the LAPACK dgbtf2 / dgbtrs scheme, one thread per edge, band stored edge-fastest so
// that a warp's accesses coalesce).  Y_e = K_e^{-1} C_e gives the 4 x 4 Schur contribution S_e = -D_e Y_e;
// the bifurcation system (2 x 2 blocks {P_b, lam_b}, the network's own topology) is eliminated leaf -> root
// over the same chunk / level schedule as the P1/DG0 path -- no fill on a tree.  Graph edges that close a
// cycle keep their diagonal blocks only (the outer FGMRES absorbs the difference).
// Which entries K_e, C_e, D_e have is listed per edge type by the host (condense.py) from the reference
// element tables; their values are coef or coef * (R h)_cell with R h accumulated by the assembly, i.e.
// the factorisation is built from the same element data as A.
#pragma once

#include "precond.cuh"

namespace nxfx {

struct CondDev {
  int n_max, kl, kv, ldab;  // kv = 2 kl: super-diagonals of U after pivoting; ldab = 3 kl + 1 band rows
  int per_edge, pcell_base, pcell_stride, cont;  // cont: continuous pressure (nodal P_b exists)
  const int32_t* __restrict__ type_n;
  const int32_t* __restrict__ loc_ptr;
  const int32_t* __restrict__ loc_kind;
  const int32_t* __restrict__ loc_off;
  const int32_t* __restrict__ k_ptr;
  const int32_t* __restrict__ k_row;
  const int32_t* __restrict__ k_col;
  const int32_t* __restrict__ k_cell;
  const double* __restrict__ k_coef;
  const int32_t* __restrict__ c_ptr;
  const int32_t* __restrict__ c_row;
  const int32_t* __restrict__ c_slot;
  const double* __restrict__ c_coef;
  const int32_t* __restrict__ d_ptr;
  const int32_t* __restrict__ d_slot;
  const int32_t* __restrict__ d_col;
  const double* __restrict__ d_coef;
  const int32_t* __restrict__ bif_node;
  double* band;   // [ldab][n_max][E]
  int32_t* ipiv;  // [n_max][E]
  double* Y;      // [4][n_max][E]
  double* S;      // [16][E]
  double* y0;     // [n_max][E]
  double* h;      // [4][E]
  double* bd0;    // block tree, schedule order, 2 x 2 row-major: assembled diagonal blocks
  double* bU;     // A(t, parent)
  double* bL;     // A(parent, t)
  double* bDinv;  // inverse of the eliminated pivot block
  double* bG;     // Dinv U
  double* bH;     // L Dinv
  double* br;     // [n_bif][2]
  double* bz;     // [n_bif][2]
};

struct EdgeInfo {
  int slot, u, v, lu, lv, type, n;
};
__device__ __forceinline__ EdgeInfo cond_edge(const Net& g, const CondDev& c, int e) {
  EdgeInfo i;
  i.slot = g.edge_slot[e];
  const int4 t = g.slot_uvl[i.slot];
  i.u = t.x; i.v = t.y; i.lu = t.z; i.lv = t.w;
  i.type = (t.z >= 0 ? 1 : 0) | (t.w >= 0 ? 2 : 0);
  i.n = c.type_n[i.type];
  return i;
}

// global dof of a local unknown (condense.py K_*)
__device__ __forceinline__ int cond_glob(const Net& g, const CondDev& c, int e, const EdgeInfo& i, int kind, int off) {
  switch (kind) {
    case 0: return i.slot * c.per_edge + off;
    case 1: return c.pcell_base + e * c.pcell_stride + off;
    case 2: return g.nq + g.n_nodes + e * (g.N - 1) + off;
    case 3: return g.nq + i.u;
    default: return g.nq + i.v;
  }
}

// Views with a run-time stride: one thread's band / vector either in global memory (stride = number of edges:
// a warp's accesses coalesce) or in shared memory (stride = threads per block: conflict-free).
struct BandRef {
  double* p;
  size_t s;
  int kv, n_max;
  __device__ __forceinline__ double& operator()(int i, int j) const { return p[((size_t)(kv + i - j) * n_max + j) * s]; }
};
struct VecRef {
  double* p;
  size_t s;
  __device__ __forceinline__ double& operator[](int k) const { return p[(size_t)k * s]; }
};

// dgbtf2: unblocked banded LU with partial pivoting, kl sub- and kl super-diagonals, fill up to kv = 2 kl
__device__ __forceinline__ void cond_band_lu(const BandRef& A, int n, int kl, int32_t* __restrict__ ipiv, size_t ips) {
  int ju = 0;
  for (int j = 0; j < n; ++j) {
    const int km = min(kl, n - 1 - j);
    int jp = 0;
    double best = fabs(A(j, j));
    for (int i = 1; i <= km; ++i) {
      const double a = fabs(A(j + i, j));
      if (a > best) { best = a; jp = i; }
    }
    ipiv[(size_t)j * ips] = j + jp;
    ju = max(ju, min(j + jp + kl, n - 1));  // last column the pivot row reaches
    if (jp != 0)
      for (int col = j; col <= ju; ++col) {
        const double t = A(j, col);
        A(j, col) = A(j + jp, col);
        A(j + jp, col) = t;
      }
    // (a zero pivot -- singular K_e -- propagates inf / nan: the residual check of the solve reports it)
    const double inv = 1.0 / A(j, j);
    for (int i = 1; i <= km; ++i) A(j + i, j) *= inv;
    for (int col = j + 1; col <= ju; ++col) {
      const double ujc = A(j, col);
      if (ujc != 0.0)
        for (int i = 1; i <= km; ++i) A(j + i, col) -= A(j + i, j) * ujc;
    }
  }
}

// dgbtrs (no transpose) on one vector, in place
__device__ __forceinline__ void cond_band_solve(const BandRef& A, int n, int kl, const int32_t* __restrict__ ipiv,
                                                size_t ips, const VecRef& b) {
  for (int j = 0; j < n; ++j) {
    const int l = ipiv[(size_t)j * ips];
    const double bj = b[l];
    if (l != j) { b[l] = b[j]; b[j] = bj; }
    const int lm = min(kl, n - 1 - j);
    if (bj != 0.0)
      for (int i = 1; i <= lm; ++i) b[j + i] -= A(j + i, j) * bj;
  }
  for (int j = n - 1; j >= 0; --j) {
    const double bj = b[j] / A(j, j);
    b[j] = bj;
    if (bj != 0.0)
      for (int i = max(0, j - A.kv); i < j; ++i) b[i] -= A(i, j) * bj;
  }
}

// K_e from the entry lists, banded LU with partial pivoting, Y_e = K_e^{-1} C_e, S_e = -D_e Y_e.
// The band stays in global memory (edge-fastest: coalesced, L2-resident per block of edges).  Measured: staging
// it in shared memory leaves room for 64-128 threads per SM only, and the LU -- a chain of dependent FP64
// read-modify-writes -- then has nothing to hide its latency behind: 1.9 / 7.0 ms instead of 1.8 / 4.9 ms for
// P2/P1 / P3/P2 at 524 k edges.
__global__ void __launch_bounds__(128)
cond_factor_kernel(Net g, CondDev c, const double* __restrict__ cell_rh) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= g.E) return;
  const size_t E = (size_t)g.E;
  const EdgeInfo ei = cond_edge(g, c, e);
  const int n = ei.n;
  const BandRef A{c.band + e, E, c.kv, c.n_max};
  for (int r = 0; r < c.ldab; ++r)
    for (int j = 0; j < n; ++j) A.p[((size_t)r * c.n_max + j) * A.s] = 0.0;
  for (int k = c.k_ptr[ei.type]; k < c.k_ptr[ei.type + 1]; ++k) {
    const int cell = c.k_cell[k];
    A(c.k_row[k], c.k_col[k]) += cell >= 0 ? c.k_coef[k] * cell_rh[(size_t)e * g.N + cell] : c.k_coef[k];
  }
  cond_band_lu(A, n, c.kl, c.ipiv + e, E);
  // Y = K^{-1} C column by column for the active nodal slots, S = -D Y
  double S[16];
#pragma unroll
  for (int k = 0; k < 16; ++k) S[k] = 0.0;
#pragma unroll
  for (int s = 0; s < 4; ++s) {
    const VecRef yv{c.Y + (size_t)s * c.n_max * E + e, E};  // column s of Y_e, solved in place
    const bool active = ((s < 2 ? ei.lu : ei.lv) >= 0) && ((s & 1) || c.cont);
    for (int k = 0; k < n; ++k) yv[k] = 0.0;
    if (!active) continue;
    for (int k = c.c_ptr[ei.type]; k < c.c_ptr[ei.type + 1]; ++k)
      if (c.c_slot[k] == s) yv[c.c_row[k]] += c.c_coef[k];
    cond_band_solve(A, n, c.kl, c.ipiv + e, E, yv);
    for (int k = c.d_ptr[ei.type]; k < c.d_ptr[ei.type + 1]; ++k) {
      const int a = c.d_slot[k];
      const double t = c.d_coef[k] * yv[c.d_col[k]];
#pragma unroll
      for (int aa = 0; aa < 4; ++aa)
        if (aa == a) S[aa * 4 + s] -= t;
    }
  }
#pragma unroll
  for (int k = 0; k < 16; ++k) c.S[(size_t)k * E + e] = S[k];
}

// The same factorisation with G lanes per edge (G = 8, 16 or 32; 256 / G edges per block), band, Y_e and pivots of
// the edge in shared memory.  Every lane of a group follows the same control flow -- the pivot search is done
// redundantly by all of them from the same shared-memory column (a broadcast) -- and the row swap, the scaling and
// the rank-1 update of a step are spread over the lanes, separated by __syncwarp().  The four columns of Y_e are
// solved at once (lane = column + 4 * helper; the helpers share the inner updates).  Same operations on the same
// operands as cond_band_lu / cond_band_solve (checked phase by phase, including read / write hazards between
// lanes, by the lock-step emulation in tests/test_condensation_lockstep.py):
// identical pivots and factors.  Against the thread-per-edge kernel
// this keeps ~768 threads per SM busy on ~100 edges instead of 128 threads on 128 edges (shared memory) or an L2
// round trip per operand (global memory).
__host__ __device__ constexpr int cond_group_smem_doubles(int ldab, int n_max) {
  return ((ldab + 4) * n_max + (n_max + 1) / 2) | 1;  // band, 4 columns of Y, pivots (ints); odd: spreads the banks
}

template <int G>
__global__ void __launch_bounds__(256)
cond_factor_group_kernel(Net g, CondDev c, const double* __restrict__ cell_rh) {
  extern __shared__ __align__(16) double cond_sm[];
  constexpr int EPB = 256 / G, H = G / 4;
  const int lane = threadIdx.x % G, grp = threadIdx.x / G;
  const int e_raw = blockIdx.x * EPB + grp;
  const bool valid = e_raw < g.E;  // a group beyond the last edge repeats it without storing: uniform control flow
  const int e = valid ? e_raw : g.E - 1;
  const size_t E = (size_t)g.E;
  const EdgeInfo ei = cond_edge(g, c, e);
  const int n = ei.n, n_max = c.n_max, kl = c.kl, kv = c.kv;
  double* __restrict__ Bd = cond_sm + (size_t)grp * cond_group_smem_doubles(c.ldab, n_max);
  double* __restrict__ Yb = Bd + c.ldab * n_max;
  int* __restrict__ piv = reinterpret_cast<int*>(Yb + 4 * n_max);
  auto A = [&](int i, int j) -> double& { return Bd[(kv + i - j) * n_max + j]; };
  for (int k = lane; k < (c.ldab + 4) * n_max; k += G) Bd[k] = 0.0;
  __syncwarp();
  // at most two entries per position (adjacent cells): their sum does not depend on the order they arrive in
  for (int k = c.k_ptr[ei.type] + lane; k < c.k_ptr[ei.type + 1]; k += G) {
    const int cell = c.k_cell[k];
    atomicAdd(&A(c.k_row[k], c.k_col[k]), cell >= 0 ? c.k_coef[k] * cell_rh[(size_t)e * g.N + cell] : c.k_coef[k]);
  }
  for (int k = c.c_ptr[ei.type] + lane; k < c.c_ptr[ei.type + 1]; k += G)
    atomicAdd(&Yb[c.c_slot[k] * n_max + c.c_row[k]], c.c_coef[k]);
  __syncwarp();
  // ---- LU (dgbtf2), one elimination step per iteration ----
  int ju = 0;
  for (int j = 0; j < n_max; ++j) {
    const bool act = j < n;
    int km = 0, jp = 0;
    if (act) {
      km = min(kl, n - 1 - j);
      double best = fabs(A(j, j));
      for (int i = 1; i <= km; ++i) {
        const double a = fabs(A(j + i, j));
        if (a > best) { best = a; jp = i; }
      }
      ju = max(ju, min(j + jp + kl, n - 1));
      if (lane == 0) {
        piv[j] = j + jp;
        if (valid) c.ipiv[(size_t)j * E + e] = j + jp;
      }
    }
    __syncwarp();  // every lane has read the column before the swap moves it
    if (act && jp != 0)
      for (int col = j + lane; col <= ju; col += G) {
        const double t = A(j, col);
        A(j, col) = A(j + jp, col);
        A(j + jp, col) = t;
      }
    __syncwarp();
    if (act) {
      const double inv = 1.0 / A(j, j);
      for (int i = 1 + lane; i <= km; i += G) A(j + i, j) *= inv;
    }
    __syncwarp();
    if (act) {
      const int total = km * (ju - j);
      for (int idx = lane; idx < total; idx += G) {
        const int i = 1 + idx % km, col = j + 1 + idx / km;
        A(j + i, col) -= A(j + i, j) * A(j, col);
      }
    }
    __syncwarp();
  }
  // ---- Y = K^{-1} C: the four columns at once ----
  const int s = lane & 3, h = lane >> 2;
  const bool col_on = ((s < 2 ? ei.lu : ei.lv) >= 0) && ((s & 1) || c.cont);
  double* __restrict__ y = Yb + s * n_max;
  for (int j = 0; j < n_max; ++j) {
    const bool act = j < n && col_on;
    int l = j;
    double bj = 0.0, tj = 0.0;
    if (act) { l = piv[j]; bj = y[l]; tj = y[j]; }
    __syncwarp();
    if (act && h == 0 && l != j) { y[l] = tj; y[j] = bj; }
    __syncwarp();
    if (act && bj != 0.0) {
      const int lm = min(kl, n - 1 - j);
      for (int i = 1 + h; i <= lm; i += H) y[j + i] -= A(j + i, j) * bj;
    }
    __syncwarp();
  }
  for (int j = n_max - 1; j >= 0; --j) {
    const bool act = j < n && col_on;
    double bj = 0.0;
    if (act) bj = y[j] / A(j, j);
    __syncwarp();
    if (act) {
      if (h == 0) y[j] = bj;
      if (bj != 0.0)
        for (int i = max(0, j - kv) + h; i < j; i += H) y[i] -= A(i, j) * bj;
    }
    __syncwarp();
  }
  // ---- S = -D Y, factors and Y to global memory (edge-fastest: the groups of a warp fill whole sectors) ----
  for (int idx = lane; idx < 16; idx += G) {
    const int a = idx >> 2, sc = idx & 3;
    double acc = 0.0;
    for (int k = c.d_ptr[ei.type]; k < c.d_ptr[ei.type + 1]; ++k)
      if (c.d_slot[k] == a) acc -= c.d_coef[k] * Yb[sc * n_max + c.d_col[k]];
    if (valid) c.S[(size_t)idx * E + e] = acc;
  }
  if (valid) {
    for (int k = lane; k < c.ldab * n_max; k += G)
      if (k % n_max < n) c.band[(size_t)k * E + e] = Bd[k];
    for (int k = lane; k < 4 * n_max; k += G)
      if (k % n_max < n) c.Y[(size_t)k * E + e] = Yb[k];
  }
}

// y0 = K_e^{-1} r_loc, h_e = D_e y0 (SMEM: the right-hand side is solved in shared memory -- n_max doubles per
// thread, full occupancy; 298 instead of 335 us for P2/P1 at 524 k edges)
template <bool SMEM>
__global__ void __launch_bounds__(128)
cond_edge_rhs_kernel(Net g, CondDev c, const double* __restrict__ r) {
  extern __shared__ __align__(16) double cond_sm[];
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= g.E) return;
  const size_t E = (size_t)g.E, T = blockDim.x;
  const EdgeInfo ei = cond_edge(g, c, e);
  const int l0 = c.loc_ptr[ei.type];
  const BandRef G{c.band + e, E, c.kv, c.n_max};
  const VecRef y{SMEM ? cond_sm + threadIdx.x : c.y0 + e, SMEM ? T : E};
  for (int k = 0; k < ei.n; ++k) y[k] = r[cond_glob(g, c, e, ei, c.loc_kind[l0 + k], c.loc_off[l0 + k])];
  cond_band_solve(G, ei.n, c.kl, c.ipiv + e, E, y);
  if (SMEM)
    for (int k = 0; k < ei.n; ++k) c.y0[(size_t)k * E + e] = y[k];
  double h[4] = {0.0, 0.0, 0.0, 0.0};
  for (int k = c.d_ptr[ei.type]; k < c.d_ptr[ei.type + 1]; ++k) {
    const int a = c.d_slot[k];
    const double t = c.d_coef[k] * y[c.d_col[k]];
#pragma unroll
    for (int aa = 0; aa < 4; ++aa)
      if (aa == a) h[aa] += t;
  }
#pragma unroll
  for (int a = 0; a < 4; ++a) c.h[(size_t)a * E + e] = h[a];
}

// Nodal blocks, one thread per bifurcation.  FACTOR: diagonal block = sum of the incident S_e blocks (in
// incidence order: deterministic), coupling blocks to the parent from the link edge.  Else: right-hand side
// r_z - sum D_e y0.  lam_w (partitioned network, else nullptr): weight of this rank's copy of a multiplier row
// of r (replicated rows count on their owner only); the nodal pressure rows are read unweighted (additive).
template <bool FACTOR>
__global__ void __launch_bounds__(kThreads)
cond_node_kernel(Net g, TreeDev t, CondDev c, const double* __restrict__ r, const double* __restrict__ lam_w = nullptr) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= g.n_bif) return;
  const size_t E = (size_t)g.E;
  const int n = t.t_of_bif[b];
  if (FACTOR) {
    double d[4] = {0.0, 0.0, 0.0, 0.0};
    for (int k = g.bif_ptr[b]; k < g.bif_ptr[b + 1]; ++k) {
      const int inc = g.bif_inc[k];
      const int e = inc >> 1, o = (inc & 1) ? 10 : 0;  // in-edge: this node is v (block rows / columns 2, 3)
      d[0] += c.S[(size_t)(o + 0) * E + e];
      d[1] += c.S[(size_t)(o + 1) * E + e];
      d[2] += c.S[(size_t)(o + 4) * E + e];
      d[3] += c.S[(size_t)(o + 5) * E + e];
    }
    if (!c.cont) { d[0] = 1.0; d[1] = 0.0; d[2] = 0.0; }  // no nodal pressure: identity placeholder
    const int pe = t.t_pedge[n];
    double U[4] = {0.0, 0.0, 0.0, 0.0}, L[4] = {0.0, 0.0, 0.0, 0.0};
    if (pe >= 0) {
      const int4 uv = g.slot_uvl[g.edge_slot[pe]];
      const bool is_u = uv.z == b;
      const int ou = is_u ? 2 : 8, ol = is_u ? 8 : 2;  // S[u-rows, v-cols] starts at 2, S[v-rows, u-cols] at 8
#pragma unroll
      for (int i = 0; i < 2; ++i)
#pragma unroll
        for (int j = 0; j < 2; ++j) {
          U[2 * i + j] = c.S[(size_t)(ou + 4 * i + j) * E + pe];
          L[2 * i + j] = c.S[(size_t)(ol + 4 * i + j) * E + pe];
        }
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      c.bd0[4 * (size_t)n + k] = d[k];
      c.bU[4 * (size_t)n + k] = U[k];
      c.bL[4 * (size_t)n + k] = L[k];
    }
  } else {
    double r0 = c.cont ? r[g.nq + c.bif_node[b]] : 0.0, r1 = lam_w ? lam_w[b] * r[g.loff + b] : r[g.loff + b];
    for (int k = g.bif_ptr[b]; k < g.bif_ptr[b + 1]; ++k) {
      const int inc = g.bif_inc[k];
      const int e = inc >> 1, o = (inc & 1) ? 2 : 0;
      r0 -= c.h[(size_t)(o + 0) * E + e];
      r1 -= c.h[(size_t)(o + 1) * E + e];
    }
    c.br[2 * (size_t)n] = c.cont ? r0 : 0.0;
    c.br[2 * (size_t)n + 1] = r1;
  }
}

struct M2 {
  double a, b, c, d;  // [[a, b], [c, d]]
};
__device__ __forceinline__ M2 ld2(const double* p, size_t n) { return M2{p[4 * n], p[4 * n + 1], p[4 * n + 2], p[4 * n + 3]}; }
__device__ __forceinline__ void st2(double* p, size_t n, M2 m) { p[4 * n] = m.a; p[4 * n + 1] = m.b; p[4 * n + 2] = m.c; p[4 * n + 3] = m.d; }
__device__ __forceinline__ M2 mul2(M2 x, M2 y) {
  return M2{x.a * y.a + x.b * y.c, x.a * y.b + x.b * y.d, x.c * y.a + x.d * y.c, x.c * y.b + x.d * y.d};
}

// Block version of tree_sweep_kernel: one thread block per chunk, level by level.
// MODE 0: factor   D_n = d0_n - sum_children H_c U_c,  Dinv_n,  G_n = Dinv_n U_n,  H_n = L_n Dinv_n
// MODE 1: forward  r_n -= sum_children H_c r_c
// MODE 2: backward z_n = Dinv_n r_n - G_n z_parent
// MODE 3: forward then backward (top chunk)
template <int MODE>
__global__ void __launch_bounds__(1024)
btree_sweep_kernel(TreeDev t, CondDev c, int chunk0) {
  const int chunk = chunk0 + blockIdx.x;
  const int L0 = t.chunk_lptr[chunk], L1 = t.chunk_lptr[chunk + 1];
  if (MODE == 0 || MODE == 1 || MODE == 3) {
    for (int L = L1 - 1; L >= L0; --L) {
      const int b = t.lvl_ptr[L], e = t.lvl_ptr[L + 1];
      for (int n = b + threadIdx.x; n < e; n += blockDim.x) {
        const int c0 = t.t_cptr[n], c1 = t.t_cptr[n + 1];
        if (MODE == 0) {
          M2 D = ld2(c.bd0, n);
          for (int k = c0; k < c1; ++k) {
            const int ch = t.t_cidx[k];
            const M2 p = mul2(ld2(c.bH, ch), ld2(c.bU, ch));
            D.a -= p.a; D.b -= p.b; D.c -= p.c; D.d -= p.d;
          }
          const double idet = 1.0 / (D.a * D.d - D.b * D.c);
          const M2 Di{D.d * idet, -D.b * idet, -D.c * idet, D.a * idet};
          st2(c.bDinv, n, Di);
          st2(c.bG, n, mul2(Di, ld2(c.bU, n)));
          st2(c.bH, n, mul2(ld2(c.bL, n), Di));
        } else {
          double r0 = c.br[2 * (size_t)n], r1 = c.br[2 * (size_t)n + 1];
          for (int k = c0; k < c1; ++k) {
            const int ch = t.t_cidx[k];
            const M2 H = ld2(c.bH, ch);
            const double s0 = c.br[2 * (size_t)ch], s1 = c.br[2 * (size_t)ch + 1];
            r0 -= H.a * s0 + H.b * s1;
            r1 -= H.c * s0 + H.d * s1;
          }
          c.br[2 * (size_t)n] = r0;
          c.br[2 * (size_t)n + 1] = r1;
        }
      }
      __syncthreads();
    }
  }
  if (MODE == 2 || MODE == 3) {
    for (int L = L0; L < L1; ++L) {
      const int b = t.lvl_ptr[L], e = t.lvl_ptr[L + 1];
      for (int n = b + threadIdx.x; n < e; n += blockDim.x) {
        const int p = t.t_parent[n];
        const M2 Di = ld2(c.bDinv, n);
        const double r0 = c.br[2 * (size_t)n], r1 = c.br[2 * (size_t)n + 1];
        double z0 = Di.a * r0 + Di.b * r1, z1 = Di.c * r0 + Di.d * r1;
        if (p >= 0) {
          const M2 G = ld2(c.bG, n);
          const double p0 = c.bz[2 * (size_t)p], p1 = c.bz[2 * (size_t)p + 1];
          z0 -= G.a * p0 + G.b * p1;
          z1 -= G.c * p0 + G.d * p1;
        }
        c.bz[2 * (size_t)n] = z0;
        c.bz[2 * (size_t)n + 1] = z1;
      }
      __syncthreads();
    }
  }
}

// Top chunk of a partitioned network, split around the caller's all-reduce (block version of tree_top_kernel's
// kPartial / kFinish, precond.cuh).  sh_idx[i]: position k of top-chunk node b0 + i in the exchanged order of the
// shared nodes (identical on every rank), -1 for a node private to this rank (sh_idx == nullptr: no shared node).
// Payload, nt = max(n_shared, 1):
//   FACTOR: partial diagonal block D_k at buf[4k], coupling blocks U_k (to the parent) at buf[4nt + 4k] and
//           L_k (from the parent) at buf[8nt + 4k], 2 x 2 row-major -- 12 nt doubles;
//   SOLVE:  partial nodal right-hand side at buf[2k] -- 2 nt doubles.
// A shared node's coupling blocks come from the edge to its shared parent, which lives on rank 0 (partition_tree):
// the other ranks contribute zeros and the sum broadcasts them.
// kPartial eliminates the private nodes (a private node has private children or bottom-chunk roots only), folds
// them and this rank's bottom-chunk roots into their shared parents and packs the shared nodes.
// kFinish reads nothing but the all-reduced payload and what it computes from it: the shared children of a shared
// node are folded in their exchanged order, so every rank performs the same operations in the same order and
// writes bit-identical factors and nodal unknowns.  The DG0 identity placeholder on the P slot (cond_node_kernel)
// arrives summed over the ranks and is set again here.  SOLVE kFinish then runs the backward sweep of the top chunk.
template <bool FACTOR, int PHASE>
__global__ void __launch_bounds__(1024)
btree_top_split_kernel(TreeDev t, CondDev c, int chunk, const int32_t* __restrict__ sh_idx, int nt, double* __restrict__ buf) {
  const int L0 = t.chunk_lptr[chunk], L1 = t.chunk_lptr[chunk + 1];
  const int b0 = t.lvl_ptr[L0];
  auto kof = [&](int n) { return (sh_idx && n >= b0) ? sh_idx[n - b0] : -1; };  // n < b0: a bottom-chunk root
  for (int L = L1 - 1; L >= L0; --L) {
    const int lb = t.lvl_ptr[L], le = t.lvl_ptr[L + 1];
    for (int n = lb + threadIdx.x; n < le; n += blockDim.x) {
      const int k = kof(n);
      if (PHASE == kFinish && k < 0) continue;  // private: complete after kPartial
      const int c0 = t.t_cptr[n], c1 = t.t_cptr[n + 1];
      if (FACTOR) {
        M2 D = PHASE == kFinish ? ld2(buf, k) : ld2(c.bd0, n);
        auto fold = [&](int ch) {
          const M2 p = mul2(ld2(c.bH, ch), ld2(c.bU, ch));
          D.a -= p.a; D.b -= p.b; D.c -= p.c; D.d -= p.d;
        };
        if (PHASE == kPartial) {
          for (int q = c0; q < c1; ++q)
            if (kof(t.t_cidx[q]) < 0) fold(t.t_cidx[q]);
          if (k >= 0) {
            st2(buf, k, D);
            st2(buf + 4 * (size_t)nt, k, ld2(c.bU, n));
            st2(buf + 8 * (size_t)nt, k, ld2(c.bL, n));
            continue;
          }
        } else {
          for (int last = -1;;) {  // shared children in exchanged order
            int best = 0x7fffffff, bc = -1;
            for (int q = c0; q < c1; ++q) {
              const int kc = kof(t.t_cidx[q]);
              if (kc > last && kc < best) { best = kc; bc = t.t_cidx[q]; }
            }
            if (bc < 0) break;
            fold(bc);
            last = best;
          }
          if (!c.cont) { D.a = 1.0; D.b = 0.0; D.c = 0.0; }
          st2(c.bU, n, ld2(buf + 4 * (size_t)nt, k));
          st2(c.bL, n, ld2(buf + 8 * (size_t)nt, k));
        }
        const double idet = 1.0 / (D.a * D.d - D.b * D.c);
        const M2 Di{D.d * idet, -D.b * idet, -D.c * idet, D.a * idet};
        st2(c.bDinv, n, Di);
        st2(c.bG, n, mul2(Di, ld2(c.bU, n)));
        st2(c.bH, n, mul2(ld2(c.bL, n), Di));
      } else {
        double r0, r1;
        if (PHASE == kFinish) { r0 = buf[2 * (size_t)k]; r1 = buf[2 * (size_t)k + 1]; }
        else { r0 = c.br[2 * (size_t)n]; r1 = c.br[2 * (size_t)n + 1]; }
        auto fold = [&](int ch) {
          const M2 H = ld2(c.bH, ch);
          const double s0 = c.br[2 * (size_t)ch], s1 = c.br[2 * (size_t)ch + 1];
          r0 -= H.a * s0 + H.b * s1;
          r1 -= H.c * s0 + H.d * s1;
        };
        if (PHASE == kPartial) {
          for (int q = c0; q < c1; ++q)
            if (kof(t.t_cidx[q]) < 0) fold(t.t_cidx[q]);
          if (k >= 0) { buf[2 * (size_t)k] = r0; buf[2 * (size_t)k + 1] = r1; continue; }
        } else {
          for (int last = -1;;) {
            int best = 0x7fffffff, bc = -1;
            for (int q = c0; q < c1; ++q) {
              const int kc = kof(t.t_cidx[q]);
              if (kc > last && kc < best) { best = kc; bc = t.t_cidx[q]; }
            }
            if (bc < 0) break;
            fold(bc);
            last = best;
          }
        }
        c.br[2 * (size_t)n] = r0;
        c.br[2 * (size_t)n + 1] = r1;
      }
    }
    __syncthreads();
  }
  if (FACTOR || PHASE != kFinish) return;
  for (int L = L0; L < L1; ++L) {  // backward sweep of the whole top chunk (as btree_sweep_kernel MODE 2)
    const int lb = t.lvl_ptr[L], le = t.lvl_ptr[L + 1];
    for (int n = lb + threadIdx.x; n < le; n += blockDim.x) {
      const int p = t.t_parent[n];
      const M2 Di = ld2(c.bDinv, n);
      const double r0 = c.br[2 * (size_t)n], r1 = c.br[2 * (size_t)n + 1];
      double z0 = Di.a * r0 + Di.b * r1, z1 = Di.c * r0 + Di.d * r1;
      if (p >= 0) {
        const M2 G = ld2(c.bG, n);
        const double p0 = c.bz[2 * (size_t)p], p1 = c.bz[2 * (size_t)p + 1];
        z0 -= G.a * p0 + G.b * p1;
        z1 -= G.c * p0 + G.d * p1;
      }
      c.bz[2 * (size_t)n] = z0;
      c.bz[2 * (size_t)n + 1] = z1;
    }
    __syncthreads();
  }
}

// Partitioned network, continuous pressure: the nodal pressure rows nq + node of the shared bifurcations
// (packed after the multiplier rows, in the exchanged order)
__global__ void __launch_bounds__(kThreads)
pack_nodal_kernel(int n_shared, int nq, const int32_t* __restrict__ shared_lm, const int32_t* __restrict__ bif_node,
                  const double* __restrict__ v, double* __restrict__ buf) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n_shared) buf[i] = v[nq + bif_node[shared_lm[i]]];
}

// After the all-reduce of [lam rows of r | (cont) P rows of r | (cont) P rows of b | ||r||^2 | ||b||^2] (the norm
// partials without any shared row): multiplier rows back into r replicated, nodal pressure rows back into r on the
// owner only (lam_weight) -- the nodal right-hand side reads them unweighted, so they must sum to the full row --
// and the norms with every shared row counted once (identical on every rank).  One block.
__global__ void __launch_bounds__(kThreads)
cond_residual_finish_kernel(int n_shared, int loff, int nq, int cont, const int32_t* __restrict__ shared_lm,
                            const int32_t* __restrict__ bif_node, const double* __restrict__ lam_weight,
                            const double* __restrict__ buf, double* __restrict__ r, double* __restrict__ nrm_out) {
  __shared__ double red[kThreads / 32];
  double ar = 0.0, ab = 0.0;
  for (int i = threadIdx.x; i < n_shared; i += blockDim.x) {
    const int lm = shared_lm[i];
    const double v = buf[i];
    r[loff + lm] = v;
    ar += v * v;
    if (cont) {
      const double p = buf[n_shared + i], pb = buf[2 * n_shared + i];
      r[nq + bif_node[lm]] = lam_weight[lm] * p;
      ar += p * p;
      ab += pb * pb;
    }
  }
  const int nr = cont ? 3 * n_shared : n_shared;
  ar = block_sum<kThreads>(ar, red);
  ab = block_sum<kThreads>(ab, red);
  if (threadIdx.x == 0) {
    nrm_out[0] = buf[nr] + ar;
    nrm_out[1] = buf[nr + 1] + ab;
  }
}

// x_loc = y0 - Y_e z_e on every edge; nodal unknowns to their global rows
template <bool ADD>
__global__ void __launch_bounds__(128)
cond_backsub_kernel(Net g, TreeDev t, CondDev c, double* __restrict__ z) {
  const int tid = blockIdx.x * blockDim.x + threadIdx.x;
  const size_t E = (size_t)g.E;
  if (tid < g.E) {
    const int e = tid;
    const EdgeInfo ei = cond_edge(g, c, e);
    double ze[4] = {0.0, 0.0, 0.0, 0.0};
    if (ei.lu >= 0) { const int n = t.t_of_bif[ei.lu]; ze[0] = c.bz[2 * (size_t)n]; ze[1] = c.bz[2 * (size_t)n + 1]; }
    if (ei.lv >= 0) { const int n = t.t_of_bif[ei.lv]; ze[2] = c.bz[2 * (size_t)n]; ze[3] = c.bz[2 * (size_t)n + 1]; }
    const int l0 = c.loc_ptr[ei.type];
    for (int k = 0; k < ei.n; ++k) {
      double v = c.y0[(size_t)k * E + e];
#pragma unroll
      for (int s = 0; s < 4; ++s) v -= c.Y[((size_t)s * c.n_max + k) * E + e] * ze[s];
      const int gi = cond_glob(g, c, e, ei, c.loc_kind[l0 + k], c.loc_off[l0 + k]);
      if (ADD) z[gi] += v; else z[gi] = v;
    }
  } else if (tid < g.E + g.n_bif) {
    const int b = tid - g.E;
    const int n = t.t_of_bif[b];
    if (c.cont) {
      const int gi = g.nq + c.bif_node[b];
      if (ADD) z[gi] += c.bz[2 * (size_t)n]; else z[gi] = c.bz[2 * (size_t)n];
    }
    if (ADD) z[g.loff + b] += c.bz[2 * (size_t)n + 1]; else z[g.loff + b] = c.bz[2 * (size_t)n + 1];
  }
}


// R*h per cell of the table-driven assembly (natural cell order), accumulated with the values
template <bool ACC>
__global__ void __launch_bounds__(kThreads)
cell_rh_generic_kernel(int64_t nc, const double* __restrict__ cell_h, const double* __restrict__ R_cell, double R_const,
                       double* __restrict__ cell_rh) {
  for (int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; k < nc; k += (int64_t)gridDim.x * blockDim.x) {
    const double v = __dmul_rn(R_cell ? R_cell[k] : R_const, cell_h[k]);
    if (ACC) cell_rh[k] += v; else cell_rh[k] = v;
  }
}

}  // namespace nxfx
