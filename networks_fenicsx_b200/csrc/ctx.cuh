// Context, error handling and device-buffer helpers of libnxfx_b200 (sm_100a, FP64).
#pragma once

#include <cuda_runtime.h>

#include <cstdarg>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/nxfx_b200.h"

namespace nxfx {

constexpr int kTileRows = 256;     // rows per thread block in the row-tiled kernels
constexpr int kTileCap = 2048;     // CSR entries staged in shared memory per tile
constexpr int kThreads = 256;

template <typename T>
struct DevBuf {
  T* p = nullptr;
  size_t n = 0;
  cudaError_t alloc(size_t count) {
    release();
    n = count;
    if (count == 0) return cudaSuccess;
    return cudaMalloc(reinterpret_cast<void**>(&p), count * sizeof(T));
  }
  void release() {
    if (p) cudaFree(p);
    p = nullptr;
    n = 0;
  }
  ~DevBuf() { release(); }
};

struct TreeSchedule {
  bool set = false;
  int n_chunks = 0, n_lvl_ptr = 0, n_chords = 0, n_top = 0;  // n_top: nodes of the (local) top chunk
  int top_b0 = 0;                     // first schedule index of the top chunk
  std::vector<int32_t> t_of_bif_h;    // host copy (positions of the shared multipliers in the top chunk)
  std::vector<int32_t> top_lvl_h;     // level table of the top chunk (schedule indices)
  int sh_lmax = -1, pr_lmin = 0;      // level ranges of the shared / private nodes of the top chunk
  int cap = 2048;  // chunk capacity of the shared-memory sweeps
  DevBuf<int32_t> bif_of_t, chunk_desc, t_inc_ptr;
  DevBuf<int2> t_inc;
  DevBuf<double> lam_nat;
  DevBuf<int32_t> t_of_bif, t_parent, t_pedge, t_pslot, t_cptr, t_cidx, chunk_lptr, lvl_ptr, chord_edge;
  // numeric
  DevBuf<double> diag0, tg, d, gd, r, lam;  // schedule order
  bool fast_ok = false;                       // every chunk fits the shared-memory sweep kernel
  bool coop_ok = false;                       // all bottom chunks can be co-resident (single-launch solve)
  bool coop_fs_ok = false;                    // the fused factor + solve can be launched cooperatively
  int coop_fs_blocks = 0;                     // ... with at most this many co-resident blocks (more chunks: several per block)
  unsigned int epoch = 0;
};

// One system matrix on the ctx's pattern: its own value array and the per-cell R*h that the network
// Schur factorisation is built from.  The reference hands out independent PETSc Mats
// (assembly.py:354, solver.py:43); every Mat of the Python layer owns one of these.
struct MatState {
  int64_t id = 0;
  DevBuf<double> vals;     // [nnz + 8]
  DevBuf<double> cell_rh;  // [nc] sum over the accumulated assemblies of R*h (N == 1: in flux-slot order)
  bool assembled = false;
  int acc_count = 0;  // number of lhs assemblies accumulated since the last zero (ADD_VALUES)
};

// Exact condensation of the table-driven (higher-order) path (condense.cuh): per-edge-type entry lists from
// the host, per-edge banded LU factors, Schur contributions, block tree factors.
struct Condensation {
  bool set = false;
  int n_max = 0, kl = 0, per_edge = 0, pcell_base = 0, pcell_stride = 0, cont = 0;
  DevBuf<int32_t> type_n, loc_ptr, loc_kind, loc_off, k_ptr, k_row, k_col, k_cell, c_ptr, c_row, c_slot, d_ptr, d_slot,
      d_col, bif_node, ipiv;
  DevBuf<double> k_coef, c_coef, d_coef, band, Y, S, y0, h, bd0, bU, bL, bDinv, bG, bH, br, bz;
  std::vector<int32_t> bif_node_h;  // host copy (nodal pressure rows of the shared bifurcations)
};

// Peer exchange of the partitioned solve (peer.cuh): this rank's exchange buffer and the mapped
// buffers of the other ranks.
struct PeerComm {
  bool created = false, ready = false;
  bool in_process = false;      // connected by nxfx_comm_connect_local: base[] are plain device pointers
  bool shared_device = false;   // another rank of the group runs on this ctx's device
  int rank = 0, nranks = 1;
  int slot = 0;                 // doubles per (channel, parity, source)
  void* local = nullptr;        // cudaMalloc'ed, exported by cudaIpcGetMemHandle
  void* base[16] = {};          // every rank's buffer as mapped into this process (base[rank] == local)
  unsigned int epoch[2] = {0, 0};
  int* err_h = nullptr;         // mapped pinned word the kernels set when a peer does not arrive
  int* err_d = nullptr;
  DevBuf<double> lam_scratch;   // [n_bif] shared rows of a residual before the exchange
};

}  // namespace nxfx

struct nxfx_ctx {
  int device = 0;
  cudaStream_t stream = nullptr;
  std::string err;
  int64_t launches = 0;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  int sm_count = 148;

  // network
  bool has_network = false, has_pattern = false, has_pbc = false, pc_ready = false;
  bool bottom_factored = false;  // multi-GPU: nxfx_pc_setup_begin done (bottom chunks factorised)
  int32_t n_nodes = 0, E = 0, gdim = 0, N = 0, n_bif = 0, n_inc = 0;
  int64_t nv = 0, nc = 0, nq = 0, poff = 0, loff = 0, ndofs = 0, nnz = 0;
  nxfx::DevBuf<double> x;          // [nv][4] vertex records {x, y, z, p_bc} (graph nodes first)
  nxfx::DevBuf<double> pos_stage;  // [n_nodes*gdim] upload staging
  nxfx::DevBuf<int4> slot_uvl;     // [E] {u, v, lm(u), lm(v)} in slot order
  nxfx::DevBuf<int2> slot_uv;      // [E] {u, v} in slot order (N == 1 assembly)
  nxfx::DevBuf<uint32_t> bif_in_bits;  // [ceil(n_inc / 32)] in-edge flag of every incidence
  nxfx::DevBuf<int32_t> slot_edge, edge_slot, edge_u, edge_v, bif_ptr, bif_inc;
  // pattern + values
  nxfx::DevBuf<int32_t> rowptr, colidx, tile_base;
  bool pipe_ok = false;  // every row tile fits one pipeline stage
  // table-driven (higher-order) assembly
  bool generic = false;
  nxfx::DevBuf<int32_t> gen_src_id, gen_bptr, gen_bid;
  nxfx::DevBuf<double> gen_src_coef, gen_bcoef, gen_cell_h;
  nxfx::Condensation cond;  // exact condensation for the generic path (nxfx_set_condensation)
  std::vector<nxfx::MatState*> mats;  // every matrix created on the current pattern ([0] = default)
  nxfx::MatState* cur = nullptr;      // the bound matrix: target of assemble, operator of spmv / solve
  int64_t next_mat_id = 1;
  bool pc_unscaled = false;           // inside the rescaled application for a k-fold accumulated matrix
  int64_t pc_mat = -1;                // matrix the tree factors were computed from (valid iff pc_ready)
  std::vector<int32_t> edge_slot_h;   // host copy (slot of the parent link edges of the schedule)
  // solver workspace
  nxfx::TreeSchedule tree;
  nxfx::DevBuf<double> edge_g, edge_c, edge_fn;  // [E] conductance, condensed rhs, F_N
  nxfx::DevBuf<double> work;                     // krylov vectors
  nxfx::DevBuf<double> work2;                    // 2 vectors: solves with a k-fold accumulated matrix
  nxfx::DevBuf<double> scal;                     // device scalars / partials
  nxfx::DevBuf<unsigned int> ticket;  // [0] reductions, [1] tree sweeps, [2] tree epoch flag
  double* scal_h = nullptr;  // pinned mirror (mapped: kernels may store results into it)
  double* scal_h_dev = nullptr;  // its device address
  bool pdl_coop_refused = false;  // the driver refused cooperative + programmatic launch
  // multi-GPU: replicated multipliers
  int32_t n_shared = 0;
  nxfx::DevBuf<int32_t> shared_lm;
  std::vector<int32_t> shared_lm_h;
  nxfx::DevBuf<int32_t> top_sh_pos;  // [n_shared] position of every shared multiplier inside the top chunk
  nxfx::DevBuf<int32_t> top_sh_idx;  // [n_top] inverse of top_sh_pos: exchanged index of a top-chunk node, -1 = private
  nxfx::DevBuf<double> lam_weight, lam_nonshared;
  nxfx::DevBuf<double> p_nonshared;  // [n_nodes] continuous pressure: 0 on the shared bifurcations (partial rows)
  nxfx::PeerComm comm;
  uint64_t peer_on = 0;  // devices this ctx's device has peer access to (bit = ordinal; nxfx_group_sum)
  // solution mirror: pinned host copy of x that nxfx_solve fills while the residual check still runs
  double* mirror_h = nullptr;
  cudaStream_t side = nullptr;
  cudaEvent_t ev_x = nullptr;
  // e2e staging
  nxfx::DevBuf<double> e2e_pbc, e2e_b, e2e_x;
};

namespace nxfx {

inline int fail(nxfx_ctx* ctx, int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  if (ctx) ctx->err = buf;
  return code;
}

#define NXFX_CUDA(ctx, call)                                                                  \
  do {                                                                                        \
    cudaError_t _e = (call);                                                                  \
    if (_e != cudaSuccess)                                                                    \
      return nxfx::fail(ctx, NXFX_ERR_CUDA, "%s:%d: %s -> %s", __FILE__, __LINE__, #call,     \
                        cudaGetErrorString(_e));                                              \
  } while (0)

#define NXFX_REQUIRE(ctx, cond, msg)                                                          \
  do {                                                                                        \
    if (!(cond)) return nxfx::fail(ctx, NXFX_ERR_INVALID, "%s: %s", __func__, msg);           \
  } while (0)

// launch + count + check
#define NXFX_LAUNCH(ctx, kernel, grid, block, smem, ...)                                      \
  do {                                                                                        \
    kernel<<<(grid), (block), (smem), (ctx)->stream>>>(__VA_ARGS__);                          \
    (ctx)->launches++;                                                                        \
    NXFX_CUDA(ctx, cudaGetLastError());                                                       \
  } while (0)

inline int64_t cdiv(int64_t a, int64_t b) { return (a + b - 1) / b; }

}  // namespace nxfx
