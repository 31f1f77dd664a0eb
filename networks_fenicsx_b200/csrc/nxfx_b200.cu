// libnxfx_b200: C ABI of the B200-native hydraulic-network assemble+solve path.
// See include/nxfx_b200.h for the contract and the reference call sites each entry replaces.

#include <cub/device/device_scan.cuh>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cmath>
#include <cstdlib>
#include <type_traits>

#include "assemble.cuh"
#include "ctx.cuh"
#include "condense.cuh"
#include "generic.cuh"
#include "precond.cuh"
#include "spmv.cuh"

using namespace nxfx;

namespace {

constexpr int kScalPartials = 8 * kMaxPartials;  // partial sums for up to 8 fused dots
constexpr int kScalSlots = 1024;                 // device scalars after the partials

Net make_net(const nxfx_ctx* c) {
  Net g;
  g.n_nodes = c->n_nodes;
  g.E = c->E;
  g.N = c->N;
  g.n_bif = c->n_bif;
  g.nq = (int32_t)c->nq;
  g.poff = (int32_t)c->poff;
  g.loff = (int32_t)c->loff;
  g.ndofs = (int32_t)c->ndofs;
  g.div_np1 = make_fastdiv((uint32_t)c->N + 1);
  g.div_n = make_fastdiv((uint32_t)std::max(c->N, 2));
  g.slot_uvl = c->slot_uvl.p;
  g.slot_lm = c->slot_lm.p;
  g.slot_edge = c->slot_edge.p;
  g.edge_slot = c->edge_slot.p;
  g.bif_ptr = c->bif_ptr.p;
  g.bif_inc = c->bif_inc.p;
  g.x2 = reinterpret_cast<const double2*>(c->x.p);
  g.slot_uv = c->slot_uv.p;
  g.bif_in_bits = c->bif_in_bits.p;
  return g;
}

TreeDev make_tree(nxfx_ctx* c) {
  TreeDev t;
  auto& s = c->tree;
  t.t_of_bif = s.t_of_bif.p;
  t.bif_of_t = s.bif_of_t.p;
  t.chunk_desc = s.chunk_desc.p;
  t.t_inc_ptr = s.t_inc_ptr.p;
  t.t_inc = s.t_inc.p;
  t.lam_nat = s.lam_nat.p;
  t.cap = s.cap;
  t.top_sh_pos = c->top_sh_pos.p;
  t.n_sh = c->top_sh_pos.p ? c->n_shared : 0;
  t.sh_lmax = s.sh_lmax;
  t.pr_lmin = s.pr_lmin;
  t.t_parent = s.t_parent.p;
  t.t_pedge = s.t_pedge.p;
  t.t_pslot = s.t_pslot.p;
  t.t_cptr = s.t_cptr.p;
  t.t_cidx = s.t_cidx.p;
  t.chunk_lptr = s.chunk_lptr.p;
  t.lvl_ptr = s.lvl_ptr.p;
  t.diag0 = s.diag0.p;
  t.tg = s.tg.p;
  t.d = s.d.p;
  t.gd = s.gd.p;
  t.r = s.r.p;
  t.lam = s.lam.p;
  return t;
}

// descriptor of one use of exchange channel `ch` (advances its epoch); nranks = 0 without a communicator
PeerDev make_peer(nxfx_ctx* c, int ch) {
  PeerDev p = {};
  if (!c->comm.ready) return p;
  for (int r = 0; r < c->comm.nranks; ++r) p.base[r] = reinterpret_cast<unsigned long long>(c->comm.base[r]);
  p.rank = c->comm.rank;
  p.nranks = c->comm.nranks;
  p.slot = c->comm.slot;
  p.epoch = ++c->comm.epoch[ch];
  p.err = c->comm.err_d;
  return p;
}

CondDev make_cond(nxfx_ctx* ctx) {
  auto& k = ctx->cond;
  CondDev c;
  c.n_max = k.n_max; c.kl = k.kl; c.kv = 2 * k.kl; c.ldab = 3 * k.kl + 1;
  c.per_edge = k.per_edge; c.pcell_base = k.pcell_base; c.pcell_stride = k.pcell_stride; c.cont = k.cont;
  c.type_n = k.type_n.p; c.loc_ptr = k.loc_ptr.p; c.loc_kind = k.loc_kind.p; c.loc_off = k.loc_off.p;
  c.k_ptr = k.k_ptr.p; c.k_row = k.k_row.p; c.k_col = k.k_col.p; c.k_cell = k.k_cell.p; c.k_coef = k.k_coef.p;
  c.c_ptr = k.c_ptr.p; c.c_row = k.c_row.p; c.c_slot = k.c_slot.p; c.c_coef = k.c_coef.p;
  c.d_ptr = k.d_ptr.p; c.d_slot = k.d_slot.p; c.d_col = k.d_col.p; c.d_coef = k.d_coef.p;
  c.bif_node = k.bif_node.p;
  c.band = k.band.p; c.ipiv = k.ipiv.p; c.Y = k.Y.p; c.S = k.S.p; c.y0 = k.y0.p; c.h = k.h.p;
  c.bd0 = k.bd0.p; c.bU = k.bU.p; c.bL = k.bL.p; c.bDinv = k.bDinv.p; c.bG = k.bG.p; c.bH = k.bH.p;
  c.br = k.br.p; c.bz = k.bz.p;
  return c;
}

int vec_grid(const nxfx_ctx* c, int64_t n) {
  return (int)std::max<int64_t>(1, std::min<int64_t>(cdiv(n, kThreads), (int64_t)c->sm_count * 8));
}

template <typename T>
int upload(nxfx_ctx* ctx, DevBuf<T>& buf, const T* src, size_t n) {
  NXFX_CUDA(ctx, buf.alloc(n));
  if (n) NXFX_CUDA(ctx, cudaMemcpyAsync(buf.p, src, n * sizeof(T), cudaMemcpyHostToDevice, ctx->stream));
  return NXFX_OK;
}

// positions of the shared multipliers inside the top chunk (needs both the schedule and the shared list)
int update_top_shared(nxfx_ctx* ctx) {
  ctx->top_sh_pos.release();
  ctx->top_sh_idx.release();
  ctx->tree.sh_lmax = -1;
  ctx->tree.pr_lmin = 0;
  if (!ctx->tree.set || ctx->n_shared == 0 || ctx->tree.t_of_bif_h.empty()) return NXFX_OK;
  std::vector<int32_t> pos((size_t)ctx->n_shared);
  for (int32_t i = 0; i < ctx->n_shared; ++i) {
    const int32_t p = ctx->tree.t_of_bif_h[ctx->shared_lm_h[i]] - ctx->tree.top_b0;
    if (p < 0 || p >= ctx->tree.n_top)
      return fail(ctx, NXFX_ERR_INVALID, "shared multiplier %d is not in the top chunk of the schedule", ctx->shared_lm_h[i]);
    pos[i] = p;
  }
  NXFX_CUDA(ctx, ctx->top_sh_pos.alloc(pos.size()));
  NXFX_CUDA(ctx, cudaMemcpy(ctx->top_sh_pos.p, pos.data(), pos.size() * sizeof(int32_t), cudaMemcpyHostToDevice));
  std::vector<int32_t> idx((size_t)ctx->tree.n_top, -1);
  for (int32_t i = 0; i < ctx->n_shared; ++i) idx[pos[i]] = i;
  NXFX_CUDA(ctx, ctx->top_sh_idx.alloc(idx.size()));
  NXFX_CUDA(ctx, cudaMemcpy(ctx->top_sh_idx.p, idx.data(), idx.size() * sizeof(int32_t), cudaMemcpyHostToDevice));
  // level ranges: shared nodes live in levels [0, sh_lmax], private ones in [pr_lmin, nl)
  const std::vector<int32_t>& lv = ctx->tree.top_lvl_h;
  const int nl = (int)lv.size() - 1;
  std::vector<char> is_sh((size_t)ctx->tree.n_top, 0);
  for (int32_t p : pos) is_sh[p] = 1;
  ctx->tree.sh_lmax = -1;
  ctx->tree.pr_lmin = nl;
  for (int L = 0; L < nl; ++L)
    for (int n = lv[L]; n < lv[L + 1]; ++n) {
      if (is_sh[n - ctx->tree.top_b0]) ctx->tree.sh_lmax = L;
      else ctx->tree.pr_lmin = std::min(ctx->tree.pr_lmin, L);
    }
  return NXFX_OK;
}

// continuous pressure on a partitioned network: weights of the nodal pressure rows in the local norms (needs the
// shared list and the condensation tables, whichever comes last builds it)
int update_pressure_weight(nxfx_ctx* ctx) {
  ctx->p_nonshared.release();
  if (!ctx->generic || !ctx->cond.set || !ctx->cond.cont || !ctx->lam_weight.p || ctx->n_shared == 0) return NXFX_OK;
  std::vector<double> w((size_t)ctx->n_nodes, 1.0);
  for (int32_t lm : ctx->shared_lm_h) w[ctx->cond.bif_node_h[lm]] = 0.0;
  NXFX_CUDA(ctx, ctx->p_nonshared.alloc(w.size()));
  NXFX_CUDA(ctx, cudaMemcpy(ctx->p_nonshared.p, w.data(), w.size() * sizeof(double), cudaMemcpyHostToDevice));
  return NXFX_OK;
}

int ensure_scal(nxfx_ctx* ctx) {
  if (ctx->scal.p) return NXFX_OK;
  NXFX_CUDA(ctx, ctx->scal.alloc(kScalPartials + kScalSlots));
  NXFX_CUDA(ctx, cudaMemsetAsync(ctx->scal.p, 0, (kScalPartials + kScalSlots) * sizeof(double), ctx->stream));
  NXFX_CUDA(ctx, ctx->ticket.alloc(4));
  NXFX_CUDA(ctx, cudaMemsetAsync(ctx->ticket.p, 0, 4 * sizeof(unsigned int), ctx->stream));
  NXFX_CUDA(ctx, cudaHostAlloc(reinterpret_cast<void**>(&ctx->scal_h), kScalSlots * sizeof(double), cudaHostAllocMapped));
  NXFX_CUDA(ctx, cudaHostGetDevicePointer(reinterpret_cast<void**>(&ctx->scal_h_dev), ctx->scal_h, 0));
  return NXFX_OK;
}

double* slot(nxfx_ctx* ctx, int i) { return ctx->scal.p + kScalPartials + i; }

bool is_assembled(const nxfx_ctx* ctx) { return ctx->cur && ctx->cur->assembled; }

void release_matrices(nxfx_ctx* ctx) {
  for (MatState* m : ctx->mats) delete m;
  ctx->mats.clear();
  ctx->cur = nullptr;
  ctx->pc_ready = false;
  ctx->pc_mat = -1;
}

// a zeroed matrix on the current pattern
int new_matrix(nxfx_ctx* ctx, int64_t id, MatState** out) {
  auto* m = new MatState();
  m->id = id;
  ctx->mats.push_back(m);
  NXFX_CUDA(ctx, m->vals.alloc((size_t)ctx->nnz + 8));
  NXFX_CUDA(ctx, cudaMemsetAsync(m->vals.p, 0, ((size_t)ctx->nnz + 8) * sizeof(double), ctx->stream));
  NXFX_CUDA(ctx, m->cell_rh.alloc((size_t)ctx->nc));
  NXFX_CUDA(ctx, cudaMemsetAsync(m->cell_rh.p, 0, (size_t)ctx->nc * sizeof(double), ctx->stream));
  if (out) *out = m;
  return NXFX_OK;
}

// k-fold accumulation (ADD_VALUES without zeroEntries): the solver needs the count, see do_pc_apply
void note_lhs_assembled(nxfx_ctx* ctx, int accumulate) {
  MatState* m = ctx->cur;
  m->acc_count = (accumulate && m->assembled) ? m->acc_count + 1 : 1;
  m->assembled = true;
  m->static_valid = false;  // nxfx_assemble sets it again after a non-accumulating P1/DG0 assembly
  ctx->pc_ready = false;
  ctx->bottom_factored = false;
}

void bind_matrix(nxfx_ctx* ctx, MatState* m) {
  if (ctx->cur != m) ctx->bottom_factored = false;
  ctx->cur = m;
  // the tree factors belong to ONE matrix: binding another one invalidates them
  if (ctx->pc_ready && ctx->pc_mat != m->id) ctx->pc_ready = false;
}

// the factors of the preconditioner now belong to the bound matrix
void mark_factored(nxfx_ctx* ctx) {
  ctx->pc_ready = true;
  ctx->pc_mat = ctx->cur->id;
}

// callers that never create a matrix (plain C users of the ABI) work on matrix 0
int ensure_matrix(nxfx_ctx* ctx) {
  if (ctx->cur) return NXFX_OK;
  for (MatState* m : ctx->mats)
    if (m->id == 0) { bind_matrix(ctx, m); return NXFX_OK; }
  MatState* m = nullptr;
  int rc = new_matrix(ctx, 0, &m);
  if (rc) return rc;
  bind_matrix(ctx, m);
  return NXFX_OK;
}

int build_vertices(nxfx_ctx* ctx) {
  const int n3 = ctx->n_nodes * 3;
  NXFX_LAUNCH(ctx, pad_nodes_kernel, (int)cdiv(n3, kThreads), kThreads, 0, ctx->n_nodes, ctx->gdim,
              ctx->pos_stage.p, ctx->x.p);
  if (ctx->N > 1) {
    const int64_t total = (int64_t)ctx->E * (ctx->N - 1) * 3;
    NXFX_LAUNCH(ctx, interior_vertices_kernel, vec_grid(ctx, total), kThreads, 0, ctx->n_nodes,
                ctx->E, ctx->N, ctx->edge_u.p, ctx->edge_v.p, ctx->x.p);
  }
  return NXFX_OK;
}

// ---- solver building blocks ------------------------------------------------------------------
// launch shape of spmv_pipe_kernel: persistent blocks (their partials stay within kMaxPartials)
struct PipeShape {
  int ntiles, grid;
};
PipeShape pipe_shape(const nxfx_ctx* ctx) {
  const int ntiles = (int)cdiv(ctx->ndofs, kTileRows);
  return {ntiles, std::min({ntiles, ctx->sm_count * kPipeBlocksPerSM, kMaxPartials})};
}

int do_spmv(nxfx_ctx* ctx, const double* x, double* y) {
  const int ntiles = (int)cdiv(ctx->ndofs, kTileRows);
  if (ctx->pipe_ok) {
    const PipeShape ps = pipe_shape(ctx);
    NXFX_LAUNCH(ctx, spmv_pipe_kernel<0>, ps.grid, kPipeThreads, kPipeSmem, (int)ctx->ndofs, ps.ntiles,
                ctx->rowptr.p, ctx->colidx.p, ctx->cur->vals.p, ctx->tile_base.p, x, y, nullptr, nullptr,
                nullptr, nullptr);
    return NXFX_OK;
  }
  NXFX_LAUNCH(ctx, spmv_kernel<0>, ntiles, kTileRows, 0, (int)ctx->ndofs, ntiles, ctx->rowptr.p,
              ctx->colidx.p, ctx->cur->vals.p, x, y, nullptr, nullptr, nullptr, nullptr);
  return NXFX_OK;
}

// pdl: launch as programmatic dependent of the preceding kernel -- only where that kernel does not
// write the matrix (the blocks prefetch matrix tiles before they wait for it)
int do_residual(nxfx_ctx* ctx, const double* b, const double* x, double* r, double* norm2_d, bool pdl = false) {
  const int ntiles = (int)cdiv(ctx->ndofs, kTileRows);
  if (ctx->comm.ready) {
    // partitioned network: the kernel itself exchanges the shared rows and the norm partials with the
    // other ranks over NVLink; norm2_d receives the GLOBAL [||r||^2, ||b||^2], identical on all ranks
    NXFX_REQUIRE(ctx, ctx->pipe_ok && ctx->lam_nonshared.p, "the fused partitioned residual needs the pipelined SpMV and nxfx_set_shared");
    const PipeShape ps = pipe_shape(ctx);
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(ps.grid);
    cfg.blockDim = dim3(kPipeThreads);
    cfg.dynamicSmemBytes = kPipeSmem;
    cfg.stream = ctx->stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = pdl ? 1 : 0;
    NXFX_CUDA(ctx, cudaLaunchKernelEx(&cfg, spmv_pipe_kernel<3>, (int)ctx->ndofs, ps.ntiles, (const int32_t*)ctx->rowptr.p,
                                      (const int32_t*)ctx->colidx.p, (const double*)ctx->cur->vals.p,
                                      (const int32_t*)ctx->tile_base.p, x, r, b, ctx->scal.p, ctx->ticket.p, norm2_d,
                                      (int)ctx->loff, (const double*)ctx->lam_nonshared.p, (const double*)ctx->lam_weight.p,
                                      make_peer(ctx, 1), (const int32_t*)ctx->shared_lm.p, (int)ctx->n_shared,
                                      ctx->comm.lam_scratch.p));
    ctx->launches++;
    return NXFX_OK;
  }
  if (ctx->pipe_ok && !pdl) {
    const PipeShape ps = pipe_shape(ctx);
    NXFX_LAUNCH(ctx, spmv_pipe_kernel<1>, ps.grid, kPipeThreads, kPipeSmem, (int)ctx->ndofs, ps.ntiles,
                ctx->rowptr.p, ctx->colidx.p, ctx->cur->vals.p, ctx->tile_base.p, x, r, b, ctx->scal.p,
                ctx->ticket.p, norm2_d);
    return NXFX_OK;
  }
  if (ctx->pipe_ok) {
    const PipeShape ps = pipe_shape(ctx);
    // programmatic dependent launch: the blocks set up their ring and prefetch matrix tiles
    // while the preceding kernel (normally the back-substitution producing x) drains
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(ps.grid);
    cfg.blockDim = dim3(kPipeThreads);
    cfg.dynamicSmemBytes = kPipeSmem;
    cfg.stream = ctx->stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    NXFX_CUDA(ctx, cudaLaunchKernelEx(&cfg, spmv_pipe_kernel<1>, (int)ctx->ndofs, ps.ntiles, (const int32_t*)ctx->rowptr.p,
                                      (const int32_t*)ctx->colidx.p, (const double*)ctx->cur->vals.p,
                                      (const int32_t*)ctx->tile_base.p, x, r, b, ctx->scal.p, ctx->ticket.p, norm2_d, 0,
                                      (const double*)nullptr, (const double*)nullptr, PeerDev{}, (const int32_t*)nullptr, 0,
                                      (double*)nullptr));
    ctx->launches++;
    return NXFX_OK;
  }
  const int grid = std::min(ntiles, kMaxPartials);
  NXFX_LAUNCH(ctx, spmv_kernel<1>, grid, kTileRows, 0, (int)ctx->ndofs, ntiles, ctx->rowptr.p,
              ctx->colidx.p, ctx->cur->vals.p, x, r, b, ctx->scal.p, ctx->ticket.p, norm2_d);
  return NXFX_OK;
}

template <int K>
int launch_multi_dot(nxfx_ctx* ctx, int n, const double* A, size_t stride, const double* w, double* out) {
  NXFX_LAUNCH(ctx, multi_dot_kernel<K>, vec_grid(ctx, n), kThreads, 0, n, A, stride, w, ctx->scal.p,
              ctx->ticket.p, out);
  return NXFX_OK;
}

int do_multi_dot(nxfx_ctx* ctx, int n, int k, const double* A, size_t stride, const double* w, double* out) {
  int j = 0;
  while (j < k) {
    const int m = std::min(8, k - j);
    const double* Aj = A + (size_t)j * stride;
    int rc = NXFX_OK;
    switch (m) {
      case 8: rc = launch_multi_dot<8>(ctx, n, Aj, stride, w, out + j); break;
      case 7: rc = launch_multi_dot<7>(ctx, n, Aj, stride, w, out + j); break;
      case 6: rc = launch_multi_dot<6>(ctx, n, Aj, stride, w, out + j); break;
      case 5: rc = launch_multi_dot<5>(ctx, n, Aj, stride, w, out + j); break;
      case 4: rc = launch_multi_dot<4>(ctx, n, Aj, stride, w, out + j); break;
      case 3: rc = launch_multi_dot<3>(ctx, n, Aj, stride, w, out + j); break;
      case 2: rc = launch_multi_dot<2>(ctx, n, Aj, stride, w, out + j); break;
      default: rc = launch_multi_dot<1>(ctx, n, Aj, stride, w, out + j); break;
    }
    if (rc) return rc;
    j += m;
  }
  return NXFX_OK;
}

template <int K>
int launch_multi_axpy(nxfx_ctx* ctx, int n, const double* A, size_t stride, const double* h, double sign, double* w) {
  NXFX_LAUNCH(ctx, multi_axpy_kernel<K>, vec_grid(ctx, n), kThreads, 0, n, A, stride, h, sign, w);
  return NXFX_OK;
}

int do_multi_axpy(nxfx_ctx* ctx, int n, int k, const double* A, size_t stride, const double* h, double sign, double* w) {
  int j = 0;
  while (j < k) {
    const int m = std::min(8, k - j);
    const double* Aj = A + (size_t)j * stride;
    int rc = NXFX_OK;
    switch (m) {
      case 8: rc = launch_multi_axpy<8>(ctx, n, Aj, stride, h + j, sign, w); break;
      case 7: rc = launch_multi_axpy<7>(ctx, n, Aj, stride, h + j, sign, w); break;
      case 6: rc = launch_multi_axpy<6>(ctx, n, Aj, stride, h + j, sign, w); break;
      case 5: rc = launch_multi_axpy<5>(ctx, n, Aj, stride, h + j, sign, w); break;
      case 4: rc = launch_multi_axpy<4>(ctx, n, Aj, stride, h + j, sign, w); break;
      case 3: rc = launch_multi_axpy<3>(ctx, n, Aj, stride, h + j, sign, w); break;
      case 2: rc = launch_multi_axpy<2>(ctx, n, Aj, stride, h + j, sign, w); break;
      default: rc = launch_multi_axpy<1>(ctx, n, Aj, stride, h + j, sign, w); break;
    }
    if (rc) return rc;
    j += m;
  }
  return NXFX_OK;
}

inline size_t vec_stride(const nxfx_ctx* ctx);
int ensure_work(nxfx_ctx* ctx, size_t nvec);

// fused: N == 1 -- the kernels evaluate the nodes' diagonal / right-hand side themselves from
// (r, cell_rh), so the separate bif_*_n1 kernel is not launched.
int tree_pass(nxfx_ctx* ctx, bool factor, const double* fuse_r = nullptr, bool fuse = false) {
  auto& s = ctx->tree;
  TreeDev t = make_tree(ctx);
  const int nb = s.n_chunks - 1;  // bottom chunks; the last chunk is the top of the forest
  if (s.fast_ok) {
    const int grid = std::max(nb, 1);
    unsigned int* tk = ctx->ticket.p + 1;
    FusedN1 fin{make_net(ctx), nullptr, nullptr};
    if (factor) {
      if (fuse) fin.cell_rh = ctx->cur->cell_rh.p;
      NXFX_LAUNCH(ctx, tree_factor_kernel, grid, kTreeThreads, tree_smem_bytes(ctx->tree.cap), t, nb, tk, 1, fin);
    } else if (s.coop_ok && nb > 0) {
      if (fuse) { fin.r = fuse_r; fin.cell_rh = ctx->cur->cell_rh.p; }
      unsigned int* fl = ctx->ticket.p + 2;
      unsigned int ep = ++s.epoch;
      int nbv = nb;
      void* args[] = {&t, &nbv, &tk, &fl, &ep, &fin};
      NXFX_CUDA(ctx, cudaLaunchCooperativeKernel(reinterpret_cast<void*>(tree_solve_coop_kernel), dim3(nb + 1), dim3(kTreeThreads),
                                                 args, tree_smem_bytes(ctx->tree.cap), ctx->stream));
      ctx->launches++;
    } else {
      NXFX_LAUNCH(ctx, tree_solve_kernel<kTreeUp>, grid, kTreeThreads, tree_smem_bytes(ctx->tree.cap), t, nb, tk, 1);
      if (nb > 0) NXFX_LAUNCH(ctx, tree_solve_kernel<kTreeDown>, nb, kTreeThreads, tree_smem_bytes(ctx->tree.cap), t, nb, tk, 1);
    }
    return NXFX_OK;
  }
  if (factor) {
    if (nb > 0) NXFX_LAUNCH(ctx, tree_sweep_kernel<kTreeFactor>, nb, 1024, 0, t, ctx->edge_g.p, 0);
    NXFX_LAUNCH(ctx, tree_sweep_kernel<kTreeFactor>, 1, 1024, 0, t, ctx->edge_g.p, nb);
  } else {
    if (nb > 0) NXFX_LAUNCH(ctx, tree_sweep_kernel<kTreeUp>, nb, 1024, 0, t, ctx->edge_g.p, 0);
    NXFX_LAUNCH(ctx, tree_sweep_kernel<kTreeUpDown>, 1, 1024, 0, t, ctx->edge_g.p, nb);
    if (nb > 0) NXFX_LAUNCH(ctx, tree_sweep_kernel<kTreeDown>, nb, 1024, 0, t, ctx->edge_g.p, 0);
  }
  return NXFX_OK;
}

// ---- table-driven path: exact condensation (condense.cuh) ---------------------------------------
constexpr int kCondThreads = 128;
constexpr size_t kCondSmemMax = 220 * 1024;

// threads per block of the shared-memory variants (0: does not fit, use the global-memory variant)
bool cond_smem_enabled() {  // NXFX_COND_SMEM=0: global-memory variants only (A/B measurements)
  static const bool on = [] { const char* e = std::getenv("NXFX_COND_SMEM"); return !(e && e[0] == '0'); }();
  return on;
}
// lanes per edge of the cooperative factorisation: the fewest that leave room for three blocks per SM, else the
// fewest that fit at all; 0 = the edge's block does not fit shared memory even with one warp per edge
int cond_group_lanes(const nxfx_ctx* ctx) {
  static const bool on = [] { const char* e = std::getenv("NXFX_COND_GROUP"); return !(e && e[0] == '0'); }();
  if (!on) return 0;
  const size_t per_edge = (size_t)cond_group_smem_doubles(3 * ctx->cond.kl + 1, ctx->cond.n_max) * sizeof(double);
  for (int G : {8, 16, 32})
    if ((256 / G) * per_edge <= 72 * 1024) return G;
  for (int G : {8, 16, 32})
    if ((256 / G) * per_edge <= kCondSmemMax) return G;
  return 0;
}
int cond_rhs_threads(const nxfx_ctx* ctx) {
  if (!cond_smem_enabled()) return 0;
  const size_t t = std::min<size_t>(kCondThreads, kCondSmemMax / ((size_t)ctx->cond.n_max * sizeof(double))) & ~(size_t)31;
  return (int)t;
}

// everything of the factorisation below the top chunk: edge factors, nodal blocks, bottom chunks
int cond_factor_local(nxfx_ctx* ctx) {
  NXFX_REQUIRE(ctx, ctx->cond.set, "nxfx_set_condensation has not been called");
  NXFX_REQUIRE(ctx, ctx->tree.set, "nxfx_set_tree_schedule has not been called");
  Net g = make_net(ctx);
  CondDev c = make_cond(ctx);
  // G lanes per edge with the band in shared memory when an edge's block fits; else one thread per edge out of
  // global memory (very long edges).  NXFX_COND_GROUP=0 forces the latter (A/B measurements).
  const int G = cond_group_lanes(ctx);
  const size_t gsm = (size_t)cond_group_smem_doubles(c.ldab, c.n_max) * sizeof(double);
  if (G == 8) NXFX_LAUNCH(ctx, cond_factor_group_kernel<8>, (int)cdiv(ctx->E, 32), 256, 32 * gsm, g, c, ctx->cur->cell_rh.p);
  else if (G == 16) NXFX_LAUNCH(ctx, cond_factor_group_kernel<16>, (int)cdiv(ctx->E, 16), 256, 16 * gsm, g, c, ctx->cur->cell_rh.p);
  else if (G == 32) NXFX_LAUNCH(ctx, cond_factor_group_kernel<32>, (int)cdiv(ctx->E, 8), 256, 8 * gsm, g, c, ctx->cur->cell_rh.p);
  else NXFX_LAUNCH(ctx, cond_factor_kernel, (int)cdiv(ctx->E, kCondThreads), kCondThreads, 0, g, c, ctx->cur->cell_rh.p);
  if (ctx->n_bif > 0) {
    TreeDev t = make_tree(ctx);
    NXFX_LAUNCH(ctx, cond_node_kernel<true>, (int)cdiv(ctx->n_bif, kThreads), kThreads, 0, g, t, c, nullptr);
    const int nb = ctx->tree.n_chunks - 1;
    if (nb > 0) NXFX_LAUNCH(ctx, btree_sweep_kernel<kTreeFactor>, nb, 1024, 0, t, c, 0);
  }
  return NXFX_OK;
}

int do_cond_setup(nxfx_ctx* ctx) {
  int rc = cond_factor_local(ctx);
  if (rc) return rc;
  if (ctx->n_bif > 0) NXFX_LAUNCH(ctx, btree_sweep_kernel<kTreeFactor>, 1, 1024, 0, make_tree(ctx), make_cond(ctx), ctx->tree.n_chunks - 1);
  mark_factored(ctx);
  return NXFX_OK;
}

// y0, h per edge, nodal right-hand sides, forward sweep of the bottom chunks (lam_w: see cond_node_kernel)
int cond_forward_local(nxfx_ctx* ctx, const double* r, const double* lam_w) {
  Net g = make_net(ctx);
  CondDev c = make_cond(ctx);
  const int tr = cond_rhs_threads(ctx);
  if (tr > 0) {
    NXFX_LAUNCH(ctx, cond_edge_rhs_kernel<true>, (int)cdiv(ctx->E, tr), tr, (size_t)c.n_max * sizeof(double) * tr, g, c, r);
  } else {
    NXFX_LAUNCH(ctx, cond_edge_rhs_kernel<false>, (int)cdiv(ctx->E, kCondThreads), kCondThreads, 0, g, c, r);
  }
  if (ctx->n_bif > 0) {
    TreeDev t = make_tree(ctx);
    NXFX_LAUNCH(ctx, cond_node_kernel<false>, (int)cdiv(ctx->n_bif, kThreads), kThreads, 0, g, t, c, r, lam_w);
    const int nb = ctx->tree.n_chunks - 1;
    if (nb > 0) NXFX_LAUNCH(ctx, btree_sweep_kernel<kTreeUp>, nb, 1024, 0, t, c, 0);
  }
  return NXFX_OK;
}

// backward sweep of the bottom chunks, back-substitution on the edges
int cond_backward_local(nxfx_ctx* ctx, double* z, bool add) {
  Net g = make_net(ctx);
  CondDev c = make_cond(ctx);
  TreeDev t = make_tree(ctx);
  const int nb = ctx->tree.n_chunks - 1;
  if (ctx->n_bif > 0 && nb > 0) NXFX_LAUNCH(ctx, btree_sweep_kernel<kTreeDown>, nb, 1024, 0, t, c, 0);
  const int grid = (int)cdiv((int64_t)ctx->E + ctx->n_bif, kCondThreads);
  if (add) NXFX_LAUNCH(ctx, cond_backsub_kernel<true>, grid, kCondThreads, 0, g, t, c, z);
  else NXFX_LAUNCH(ctx, cond_backsub_kernel<false>, grid, kCondThreads, 0, g, t, c, z);
  return NXFX_OK;
}

int do_cond_apply(nxfx_ctx* ctx, const double* r, double* z, bool add) {
  NXFX_REQUIRE(ctx, ctx->pc_ready, "pc_setup has not been run");
  int rc = cond_forward_local(ctx, r, nullptr);
  if (rc) return rc;
  if (ctx->n_bif > 0) NXFX_LAUNCH(ctx, btree_sweep_kernel<kTreeUpDown>, 1, 1024, 0, make_tree(ctx), make_cond(ctx), ctx->tree.n_chunks - 1);
  return cond_backward_local(ctx, z, add);
}

// ---- P1/DG0 building blocks: one cell per edge (n1) or several ------------------------------------
// n1: the node and edge kernels read the cell data themselves and move the two flux dofs of an edge with
// one 16-byte access.  (The global-memory fallback sweeps of a schedule without fast_ok read edge_g.)
bool n1_kernels(const nxfx_ctx* ctx) { return ctx->N == 1 && ctx->tree.fast_ok; }

int check_aligned(nxfx_ctx* ctx, const double* r, const double* z = nullptr) {
  NXFX_REQUIRE(ctx, (reinterpret_cast<uintptr_t>(r) & 15) == 0 && (reinterpret_cast<uintptr_t>(z) & 15) == 0,
               "vectors must be 16-byte aligned");
  return NXFX_OK;
}

// diagonals of the nodes; bif = false: only what the edges contribute (the edge conductances)
int node_diag(nxfx_ctx* ctx, bool bif) {
  if (n1_kernels(ctx)) {
    if (bif) NXFX_LAUNCH(ctx, bif_diag_n1_kernel, (int)cdiv(ctx->n_bif, kThreads), kThreads, 0, make_net(ctx), make_tree(ctx), ctx->cur->cell_rh.p);
    return NXFX_OK;
  }
  NXFX_LAUNCH(ctx, edge_conductance_kernel, (int)cdiv(ctx->E, kThreads), kThreads, 0, make_net(ctx), ctx->cur->cell_rh.p, ctx->edge_g.p);
  if (bif) NXFX_LAUNCH(ctx, bif_diag_kernel, (int)cdiv(ctx->n_bif, kThreads), kThreads, 0, make_net(ctx), make_tree(ctx), ctx->edge_g.p);
  return NXFX_OK;
}

// right-hand sides of the nodes; bif = false: only the per-edge condensation
int node_rhs(nxfx_ctx* ctx, const double* r, bool bif) {
  Net g = make_net(ctx);
  TreeDev t = make_tree(ctx);
  if (n1_kernels(ctx)) {
    if (bif) NXFX_LAUNCH(ctx, bif_rhs_n1_kernel, (int)cdiv(ctx->n_bif, kThreads), kThreads, 0, g, t, r, ctx->cur->cell_rh.p, ctx->lam_weight.p);
    return NXFX_OK;
  }
  NXFX_LAUNCH(ctx, edge_condense_kernel<false>, (int)cdiv(ctx->E, kThreads), kThreads, 0, g, ctx->cur->cell_rh.p, r,
              ctx->edge_c.p, ctx->edge_fn.p, nullptr);
  if (bif)
    NXFX_LAUNCH(ctx, bif_rhs_kernel<false>, (int)cdiv(ctx->n_bif, kThreads), kThreads, 0, g, t, r, ctx->edge_g.p, ctx->edge_c.p,
                ctx->edge_fn.p, ctx->lam_weight.p);
  return NXFX_OK;
}

// z (+)= the edge unknowns from the solved nodal ones.  pdl: the n1 kernel is launched as programmatic dependent of
// the tree kernel and stages its edge data while that finishes (the general kernel has no such wait: plain launch).
int edge_backsub(nxfx_ctx* ctx, const double* r, double* z, bool add, bool pdl = false) {
  Net g = make_net(ctx);
  TreeDev t = make_tree(ctx);
  const double* cell_rh = ctx->cur->cell_rh.p;
  const int grid = (int)cdiv((int64_t)ctx->E + ctx->n_bif, kThreads);
  if (!n1_kernels(ctx)) {
    if (add) NXFX_LAUNCH(ctx, edge_backsub_kernel<true>, grid, kThreads, 0, g, t, cell_rh, r, ctx->edge_g.p, ctx->edge_c.p, z);
    else NXFX_LAUNCH(ctx, edge_backsub_kernel<false>, grid, kThreads, 0, g, t, cell_rh, r, ctx->edge_g.p, ctx->edge_c.p, z);
    return NXFX_OK;
  }
  if (!pdl) {
    if (add) NXFX_LAUNCH(ctx, edge_backsub_n1_kernel<true>, grid, kThreads, 0, g, t, cell_rh, r, z);
    else NXFX_LAUNCH(ctx, edge_backsub_n1_kernel<false>, grid, kThreads, 0, g, t, cell_rh, r, z);
    return NXFX_OK;
  }
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)grid);
  cfg.blockDim = dim3(kThreads);
  cfg.stream = ctx->stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  if (add) NXFX_CUDA(ctx, cudaLaunchKernelEx(&cfg, edge_backsub_n1_kernel<true>, g, t, cell_rh, r, z));
  else NXFX_CUDA(ctx, cudaLaunchKernelEx(&cfg, edge_backsub_n1_kernel<false>, g, t, cell_rh, r, z));
  ctx->launches++;
  return NXFX_OK;
}

int do_pc_setup(nxfx_ctx* ctx) {
  NXFX_REQUIRE(ctx, is_assembled(ctx), "assemble the matrix before pc_setup");
  if (ctx->generic) return do_cond_setup(ctx);
  NXFX_REQUIRE(ctx, ctx->tree.set, "nxfx_set_tree_schedule has not been called");
  const bool n1 = n1_kernels(ctx);
  int rc;
  if (!n1 && (rc = node_diag(ctx, ctx->n_bif > 0))) return rc;
  // n1: the factor kernel evaluates the diagonals itself
  if (ctx->n_bif > 0 && (rc = tree_pass(ctx, true, nullptr, n1))) return rc;
  mark_factored(ctx);
  return NXFX_OK;
}

// factorisation and first application z = P^{-1} r in one cooperative launch
bool can_fuse_setup(const nxfx_ctx* ctx) {
  return !ctx->generic && ctx->tree.set && ctx->tree.fast_ok && ctx->tree.coop_fs_ok && ctx->n_bif > 0 &&
         ctx->tree.n_chunks > 1 && (!ctx->lam_weight.p || ctx->comm.ready) && ctx->cur->acc_count == 1;
}

int do_pc_setup_apply(nxfx_ctx* ctx, const double* r, double* z, bool add = false) {
  NXFX_REQUIRE(ctx, is_assembled(ctx), "assemble the matrix before pc_setup");
  const bool n1 = n1_kernels(ctx);  // (can_fuse_setup: fast_ok)
  if (n1) {
    int rc = check_aligned(ctx, r, z);
    if (rc) return rc;
  }
  auto& s = ctx->tree;
  Net g = make_net(ctx);
  TreeDev t = make_tree(ctx);
  FusedN1 fin{g, r, ctx->cur->cell_rh.p, ctx->lam_weight.p};
  unsigned int* tk = ctx->ticket.p + 1;
  unsigned int* fl = ctx->ticket.p + 2;
  unsigned int ep = ++s.epoch;
  int nb = s.n_chunks - 1;
  PeerDev pc = make_peer(ctx, 0);  // multi-GPU: the top block exchanges its partial sums with the peers
  if (!n1) {
    // several cells per edge: the per-edge condensation and the bifurcation sums are separate streaming
    // kernels; the tree kernel then stages the node arrays (diag0, tg, r) instead of the incidence table
    // (two passes -- per edge, per bifurcation -- produce what the separate setup / apply kernels produce in four)
    NXFX_LAUNCH(ctx, edge_condense_kernel<true>, (int)cdiv(ctx->E, kThreads), kThreads, 0, g, ctx->cur->cell_rh.p, r,
                ctx->edge_c.p, ctx->edge_fn.p, ctx->edge_g.p);
    NXFX_LAUNCH(ctx, bif_rhs_kernel<true>, (int)cdiv(ctx->n_bif, kThreads), kThreads, 0, g, t, r, ctx->edge_g.p,
                ctx->edge_c.p, ctx->edge_fn.p, ctx->lam_weight.p);
    fin.r = nullptr;
    fin.cell_rh = nullptr;
  }
  // both kernels are programmatic dependents of their predecessor: the tree kernel stages its
  // schedule tables while the assembly drains, the back-substitution its edge data while the tree
  // kernel finishes (cooperative + programmatic launch; plain cooperative launch if refused)
  cudaLaunchConfig_t cfg = {};
  const int gb = std::min(nb, s.coop_fs_blocks - 1);  // bottom blocks (each takes ceil(nb / gb) chunks)
  cfg.gridDim = dim3(gb + 1);                         // the last block owns the top chunk
  cfg.blockDim = dim3(kTreeThreads);
  cfg.dynamicSmemBytes = tree_smem_bytes_fs(s.cap);
  cfg.stream = ctx->stream;
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeCooperative;
  attr[0].val.cooperative = 1;
  attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[1].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = ctx->pdl_coop_refused ? 1 : 2;
  const bool multi = gb < nb;
  auto kern = pc.nranks > 1 ? (multi ? tree_factor_solve_coop_kernel<true, true> : tree_factor_solve_coop_kernel<true, false>)
                            : (multi ? tree_factor_solve_coop_kernel<false, true> : tree_factor_solve_coop_kernel<false, false>);
  cudaError_t le = cudaLaunchKernelEx(&cfg, kern, t, nb, tk, fl, ep, fin, pc);
  if (le != cudaSuccess && cfg.numAttrs == 2) {
    cudaGetLastError();
    ctx->pdl_coop_refused = true;
    cfg.numAttrs = 1;
    le = cudaLaunchKernelEx(&cfg, kern, t, nb, tk, fl, ep, fin, pc);
  }
  NXFX_CUDA(ctx, le);
  ctx->launches++;
  mark_factored(ctx);
  // ranks sharing this device: a back-substitution that moved in early would hold SMs while the tree kernel
  // waits for a peer whose cooperative grid still has to become resident (DESIGN §6)
  return edge_backsub(ctx, r, z, add, !ctx->comm.shared_device);
}

int do_pc_apply(nxfx_ctx* ctx, int pc_type, const double* r, double* z, bool add = false) {
  const int n = (int)ctx->ndofs;
  if (pc_type == NXFX_PC_NETWORK_SCHUR && ctx->cur->acc_count > 1 && !ctx->pc_unscaled) {
    // The matrix holds k accumulated assemblies: A_k = [M_sum, -k B^T, k T^T; k B, 0, 0; k T, 0, 0] with
    // M_sum built from the accumulated cell_rh.  With p' = k p, lam' = k lam this is the standard
    // operator on M_sum with the constraint right-hand sides divided by k:
    //   z' = P(M_sum)^{-1} (r_q, r_p / k, r_lam / k),   z = (z'_q, z'_p / k, z'_lam / k).
    const size_t ld = vec_stride(ctx);
    if (ctx->work2.n < 2 * ld) {
      NXFX_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
      NXFX_CUDA(ctx, ctx->work2.alloc(2 * ld));
    }
    const double inv_k = 1.0 / (double)ctx->cur->acc_count;
    double* rs = ctx->work2.p;
    double* zs = ctx->work2.p + ld;
    NXFX_LAUNCH(ctx, scale_tail_kernel<false>, vec_grid(ctx, n), kThreads, 0, n, (int)ctx->poff, inv_k, r, rs);
    ctx->pc_unscaled = true;
    const int rc = do_pc_apply(ctx, pc_type, rs, zs, false);
    ctx->pc_unscaled = false;
    if (rc) return rc;
    if (add) NXFX_LAUNCH(ctx, scale_tail_kernel<true>, vec_grid(ctx, n), kThreads, 0, n, (int)ctx->poff, inv_k, zs, z);
    else NXFX_LAUNCH(ctx, scale_tail_kernel<false>, vec_grid(ctx, n), kThreads, 0, n, (int)ctx->poff, inv_k, zs, z);
    return NXFX_OK;
  }
  if (add && pc_type != NXFX_PC_NETWORK_SCHUR) {  // generic: z_tmp = P^{-1} r, z += z_tmp
    int rc = ensure_work(ctx, 3);
    if (rc) return rc;
    double* tmp = ctx->work.p + 2 * vec_stride(ctx);
    if ((rc = do_pc_apply(ctx, pc_type, r, tmp, false))) return rc;
    NXFX_LAUNCH(ctx, add_kernel, vec_grid(ctx, n), kThreads, 0, n, tmp, z);
    return NXFX_OK;
  }
  if (ctx->comm.ready) {
    // partitioned network: the stored factors of the top chunk are not kept per rank; re-eliminate with
    // the fused kernel (same cost as a solve: the sweeps are latency-bound) and exchange over NVLink
    NXFX_REQUIRE(ctx, pc_type == NXFX_PC_NETWORK_SCHUR && can_fuse_setup(ctx),
                 "the fused partitioned solve needs a forest schedule that fits the cooperative kernel and pc_type lu");
    return do_pc_setup_apply(ctx, r, z, add);
  }
  if (pc_type == NXFX_PC_NONE) {
    NXFX_CUDA(ctx, cudaMemcpyAsync(z, r, n * sizeof(double), cudaMemcpyDeviceToDevice, ctx->stream));
    return NXFX_OK;
  }
  if (pc_type == NXFX_PC_JACOBI_FLUX) {
    NXFX_LAUNCH(ctx, jacobi_flux_kernel, (int)cdiv(n, kThreads), kThreads, 0, n, (int)ctx->nq,
                ctx->rowptr.p, ctx->colidx.p, ctx->cur->vals.p, r, z);
    return NXFX_OK;
  }
  NXFX_REQUIRE(ctx, ctx->pc_ready, "pc_setup has not been run");
  if (ctx->generic) return do_cond_apply(ctx, r, z, add);
  const bool n1 = n1_kernels(ctx);
  int rc;
  if (n1 && (rc = check_aligned(ctx, r, z))) return rc;
  // n1, single-launch solve: the tree kernel evaluates the bifurcation right-hand sides itself
  const bool fuse = n1 && ctx->n_bif > 0 && ctx->tree.coop_ok && ctx->tree.n_chunks > 1 && !ctx->lam_weight.p;
  if ((rc = node_rhs(ctx, r, ctx->n_bif > 0 && !fuse))) return rc;
  if (ctx->n_bif > 0 && (rc = tree_pass(ctx, false, r, fuse))) return rc;
  return edge_backsub(ctx, r, z, add);
}

// ---- phases of the partitioned preconditioner (nxfx_pc_*_begin/_end), for either element family ----------------
// factorisation below the top chunk
int factor_bottom(nxfx_ctx* ctx) {
  if (ctx->generic) return cond_factor_local(ctx);
  int rc = node_diag(ctx, true);
  if (rc) return rc;
  const int nb = ctx->tree.n_chunks - 1;
  if (nb > 0) NXFX_LAUNCH(ctx, tree_factor_kernel, nb, kTreeThreads, tree_smem_bytes(ctx->tree.cap), make_tree(ctx), nb, ctx->ticket.p + 1, 0,
                          (FusedN1{make_net(ctx), nullptr, nullptr}));
  return NXFX_OK;
}

// nodal right-hand sides and forward sweep of the bottom chunks
int forward_bottom(nxfx_ctx* ctx, const double* r) {
  if (ctx->generic) return cond_forward_local(ctx, r, ctx->lam_weight.p);
  int rc = node_rhs(ctx, r, true);
  if (rc) return rc;
  const int nb = ctx->tree.n_chunks - 1;
  if (nb > 0) NXFX_LAUNCH(ctx, tree_solve_kernel<kTreeUp>, nb, kTreeThreads, tree_smem_bytes(ctx->tree.cap), make_tree(ctx), nb, ctx->ticket.p + 1, 0);
  return NXFX_OK;
}

// the top chunk's half of a split phase: kPartial packs this rank's partial sums of the shared nodes into buf,
// kFinish completes from the all-reduced buf (precond.cuh tree_top_split_kernel, condense.cuh btree_top_split_kernel)
template <bool FACTOR, int PHASE>
int top_split(nxfx_ctx* ctx, double* buf) {
  const int top = ctx->tree.n_chunks - 1;
  if (!ctx->generic) {
    using Op = std::conditional_t<FACTOR, FactorOp, SolveOp>;
    NXFX_LAUNCH(ctx, (tree_top_split_kernel<Op, PHASE>), 1, kTreeThreads, tree_smem_bytes(ctx->tree.cap), make_tree(ctx), top, buf,
                (FusedN1{make_net(ctx), nullptr, nullptr}));
    return NXFX_OK;
  }
  if (ctx->n_bif == 0) return NXFX_OK;
  const int32_t* idx = ctx->n_shared > 0 ? ctx->top_sh_idx.p : nullptr;
  using BlockOp = std::conditional_t<FACTOR, BlockFactor, BlockSolve>;
  NXFX_LAUNCH(ctx, (btree_top_split_kernel<BlockOp, PHASE>), 1, 1024, 0, make_tree(ctx), make_cond(ctx), top, idx,
              std::max(ctx->n_shared, 1), buf);
  return NXFX_OK;
}

// backward sweep of the bottom chunks, back-substitution on the edges
int backward_bottom(nxfx_ctx* ctx, const double* r, double* z, bool add) {
  if (ctx->generic) return cond_backward_local(ctx, z, add);
  const int nb = ctx->tree.n_chunks - 1;
  if (nb > 0) NXFX_LAUNCH(ctx, tree_solve_kernel<kTreeDown>, nb, kTreeThreads, tree_smem_bytes(ctx->tree.cap), make_tree(ctx), nb, ctx->ticket.p + 1, 0);
  return edge_backsub(ctx, r, z, add);
}

// P1/DG0 with one cell per edge: setup and first application share fused bottom and top kernels
bool fused_split(const nxfx_ctx* ctx) { return !ctx->generic && n1_kernels(ctx); }

// exchanged rows of a residual, in the order of the shared list: the multiplier rows of r, then (cont: continuous
// pressure) the nodal pressure rows of r and of b
int pack_shared(nxfx_ctx* ctx, const double* r, const double* b, double* buf, bool cont) {
  const int ns = ctx->n_shared;
  if (ns == 0) return NXFX_OK;
  NXFX_LAUNCH(ctx, pack_shared_kernel, (int)cdiv(ns, kThreads), kThreads, 0, ns, (int)ctx->loff, ctx->shared_lm.p, r, buf);
  if (!cont) return NXFX_OK;
  NXFX_LAUNCH(ctx, pack_nodal_kernel, (int)cdiv(ns, kThreads), kThreads, 0, ns, (int)ctx->nq, ctx->shared_lm.p, ctx->cond.bif_node.p,
              r, buf + ns);
  NXFX_LAUNCH(ctx, pack_nodal_kernel, (int)cdiv(ns, kThreads), kThreads, 0, ns, (int)ctx->nq, ctx->shared_lm.p, ctx->cond.bif_node.p,
              b, buf + 2 * (size_t)ns);
  return NXFX_OK;
}

// Krylov / work vectors are laid out with an EVEN stride: the N == 1 kernels read pairs of flux
// dofs with 16-byte loads, so every vector must start on a 16-byte boundary.
inline size_t vec_stride(const nxfx_ctx* ctx) { return ((size_t)ctx->ndofs + 1) & ~(size_t)1; }

int ensure_work(nxfx_ctx* ctx, size_t nvec) {
  const size_t need = nvec * vec_stride(ctx);
  if (ctx->work.n >= need) return NXFX_OK;
  NXFX_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  NXFX_CUDA(ctx, ctx->work.alloc(need));
  return NXFX_OK;
}

// sentinel of the norm words the residual kernel stores into mapped pinned memory (a NaN payload no sum of squares has)
inline double kNormSentinel() {
  const uint64_t bits = 0x7FF8DEADBEEF0001ull;
  double d;
  std::memcpy(&d, &bits, sizeof d);
  return d;
}
inline bool is_norm_sentinel(double v) {
  uint64_t bits;
  std::memcpy(&bits, &v, sizeof bits);
  return bits == 0x7FF8DEADBEEF0001ull;
}
bool poll_norms_enabled() {  // NXFX_POLL_NORMS=0: always cudaStreamSynchronize (A/B measurements)
  static const bool on = [] { const char* e = std::getenv("NXFX_POLL_NORMS"); return !(e && e[0] == '0'); }();
  return on;
}

void push_history(nxfx_solve_info* info, double v) {
  if (info->history_len < NXFX_HISTORY_LEN) info->history[info->history_len++] = v;
}

// x = P^{-1} b, then iterative refinement x += P^{-1}(b - A x) while the residual (evaluated with
// the fused norms of the SpMV kernel) exceeds refine_rtol ||b||, at most refine_steps corrections.
// The decision is taken on the host after the one synchronisation the solve needs anyway to return
// its norms: the common case (first solve already converged) costs one SpMV and no extra launch.
// refine_rtol = 0 forces every allowed correction.  The reported residual is the last one computed;
// final_residual adds an evaluation after the last correction.
// solution mirror (nxfx_set_solution_mirror): x -> pinned host memory on a side stream, ordered after what is
// enqueued on the main stream so far -- the download of the solution overlaps the residual check
int mirror_copy(nxfx_ctx* ctx, const double* x) {
  if (!ctx->mirror_h) return NXFX_OK;
  NXFX_CUDA(ctx, cudaEventRecord(ctx->ev_x, ctx->stream));
  NXFX_CUDA(ctx, cudaStreamWaitEvent(ctx->side, ctx->ev_x, 0));
  NXFX_CUDA(ctx, cudaMemcpyAsync(ctx->mirror_h, x, (size_t)ctx->ndofs * sizeof(double), cudaMemcpyDeviceToHost, ctx->side));
  return NXFX_OK;
}

int solve_preonly(nxfx_ctx* ctx, const double* b, double* x, const nxfx_solve_opts* o, nxfx_solve_info* info,
                  bool fused_setup) {
  int rc = ensure_work(ctx, 3);
  if (rc) return rc;
  double* r = ctx->work.p;
  const int steps = std::max(0, std::min(o->refine_steps, 32));
  if ((rc = fused_setup ? do_pc_setup_apply(ctx, b, x) : do_pc_apply(ctx, o->pc_type, b, x, false))) return rc;
  if ((rc = mirror_copy(ctx, x))) return rc;  // almost always the final x: corrections (below) copy again
  info->iterations = 1;
  if (steps == 0 && !o->final_residual) {  // plain preconditioner application, nothing measured
    NXFX_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    info->rhs_norm = info->residual_norm = -1.0;
    info->converged = 1;
    return NXFX_OK;
  }
  const double rt = o->refine_rtol > 0.0 ? o->refine_rtol : 0.0;
  int applied = 0;
  while (true) {
    // the reducing block stores the two norms straight into mapped pinned memory: no copy-engine hop
    // Only the norms are needed for the decision: the residual vector itself is written (by a second
    // pass, bit-identical) only if a correction follows -- never on trees.
    const bool lazy = ctx->pipe_ok;
    // the norms land in mapped pinned memory: the host watches the two words change instead of asking the driver
    // to synchronise the stream (the stream-ordered work that follows needs no host-side completion); a genuine
    // result equal to the sentinel, a faulting kernel or a long solve fall through to the synchronisation
    volatile double* nh = ctx->scal_h;
    const bool poll = poll_norms_enabled();
    if (poll) { ctx->scal_h[0] = kNormSentinel(); ctx->scal_h[1] = kNormSentinel(); }
    if ((rc = do_residual(ctx, b, x, lazy ? nullptr : r, ctx->scal_h_dev, true))) return rc;
    bool arrived = false;
    if (poll) {
      const auto t0 = std::chrono::steady_clock::now();
      for (unsigned spin = 0;; ++spin) {
        if (!is_norm_sentinel(nh[0]) && !is_norm_sentinel(nh[1])) { arrived = true; break; }
        if ((spin & 255u) == 255u && std::chrono::steady_clock::now() - t0 > std::chrono::microseconds(1500)) break;
      }
      std::atomic_thread_fence(std::memory_order_acquire);
    }
    if (!arrived) NXFX_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    info->rhs_norm = std::sqrt(ctx->scal_h[1]);
    info->residual_norm = std::sqrt(ctx->scal_h[0]);
    push_history(info, info->residual_norm);
    const bool good = std::isfinite(info->residual_norm) && info->residual_norm <= rt * info->rhs_norm;
    if (applied >= steps || (good && rt > 0.0) || !std::isfinite(info->residual_norm)) break;
    if (lazy && (rc = do_residual(ctx, b, x, r, slot(ctx, 0)))) return rc;
    if ((rc = do_pc_apply(ctx, o->pc_type, r, x, true))) return rc;
    if ((rc = mirror_copy(ctx, x))) return rc;
    ++applied;
    if (applied >= steps && !o->final_residual) break;  // residual of the iterate before the last correction
  }
  info->iterations = 1 + applied;
  const double tol = std::max(o->rtol * info->rhs_norm, o->atol);
  info->converged = std::isfinite(info->residual_norm) && info->residual_norm <= tol;
  return NXFX_OK;
}

// Right-preconditioned flexible GMRES(m), classical Gram-Schmidt with one re-orthogonalisation
// (two fused multi-dots per iteration), Givens rotations on the host: one readback per iteration.
int solve_fgmres(nxfx_ctx* ctx, const double* b, double* x, const nxfx_solve_opts* o, nxfx_solve_info* info) {
  const int n = (int)ctx->ndofs;
  const int m = std::max(1, std::min(o->restart > 0 ? o->restart : 30, 200));
  NXFX_REQUIRE(ctx, 2 * (m + 2) + 8 < kScalSlots, "restart too large");
  int rc = ensure_work(ctx, (size_t)(2 * m + 3));
  if (rc) return rc;
  const size_t ld = vec_stride(ctx);             // even: every vector is 16-byte aligned
  double* V = ctx->work.p;                       // m+1 vectors
  double* Z = V + (size_t)(m + 1) * ld;          // m vectors
  double* w = Z + (size_t)m * ld;                // 1
  double* r = w + ld;                            // 1
  double* hcol = slot(ctx, 8);                   // h[0..k], then ||w||^2
  double* hcol2 = slot(ctx, 8 + m + 2);          // second Gram-Schmidt pass
  double* ycoef = slot(ctx, 8 + 2 * (m + 2));    // solution of the small system (<= m)
  std::vector<double> H((size_t)(m + 1) * m, 0.0), cs(m), sn(m), gvec(m + 1), y(m);

  NXFX_CUDA(ctx, cudaMemsetAsync(x, 0, n * sizeof(double), ctx->stream));
  int its = 0;
  const int max_it = o->max_it > 0 ? o->max_it : 10000;
  double tol = 0.0;
  while (true) {
    if ((rc = do_residual(ctx, b, x, r, slot(ctx, 1)))) return rc;
    NXFX_CUDA(ctx, cudaMemcpyAsync(ctx->scal_h, slot(ctx, 1), 2 * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    NXFX_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    info->rhs_norm = std::sqrt(ctx->scal_h[1]);
    const double beta = std::sqrt(ctx->scal_h[0]);
    tol = std::max(o->rtol * info->rhs_norm, o->atol);
    info->residual_norm = beta;
    push_history(info, beta);
    if (!(beta > tol) || its >= max_it || !std::isfinite(beta)) break;
    NXFX_LAUNCH(ctx, scale_by_inv_norm_kernel, vec_grid(ctx, n), kThreads, 0, n, r, slot(ctx, 1), V);
    std::fill(gvec.begin(), gvec.end(), 0.0);
    gvec[0] = beta;
    int k = 0;
    for (; k < m && its < max_it; ++k, ++its) {
      double* vk = V + (size_t)k * ld;
      double* zk = Z + (size_t)k * ld;
      if ((rc = do_pc_apply(ctx, o->pc_type, vk, zk))) return rc;
      if ((rc = do_spmv(ctx, zk, w))) return rc;
      if ((rc = do_multi_dot(ctx, n, k + 1, V, ld, w, hcol))) return rc;
      if ((rc = do_multi_axpy(ctx, n, k + 1, V, ld, hcol, -1.0, w))) return rc;
      if ((rc = do_multi_dot(ctx, n, k + 1, V, ld, w, hcol2))) return rc;
      if ((rc = do_multi_axpy(ctx, n, k + 1, V, ld, hcol2, -1.0, w))) return rc;
      if ((rc = do_multi_dot(ctx, n, 1, w, 0, w, hcol + k + 1))) return rc;
      NXFX_LAUNCH(ctx, scale_by_inv_norm_kernel, vec_grid(ctx, n), kThreads, 0, n, w, hcol + k + 1,
                  V + (size_t)(k + 1) * ld);
      NXFX_CUDA(ctx, cudaMemcpyAsync(ctx->scal_h, hcol, (2 * (m + 2)) * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
      NXFX_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
      double* Hk = &H[(size_t)k * (m + 1)];
      for (int i = 0; i <= k; ++i) Hk[i] = ctx->scal_h[i] + ctx->scal_h[m + 2 + i];
      Hk[k + 1] = std::sqrt(ctx->scal_h[k + 1]);
      for (int i = 0; i < k; ++i) {
        const double t = cs[i] * Hk[i] + sn[i] * Hk[i + 1];
        Hk[i + 1] = -sn[i] * Hk[i] + cs[i] * Hk[i + 1];
        Hk[i] = t;
      }
      const double den = std::hypot(Hk[k], Hk[k + 1]);
      cs[k] = den > 0 ? Hk[k] / den : 1.0;
      sn[k] = den > 0 ? Hk[k + 1] / den : 0.0;
      Hk[k] = den;
      gvec[k + 1] = -sn[k] * gvec[k];
      gvec[k] = cs[k] * gvec[k];
      const double est = std::fabs(gvec[k + 1]);
      push_history(info, est);
      if (est <= tol || !std::isfinite(est)) { ++k; ++its; break; }
    }
    for (int i = k - 1; i >= 0; --i) {
      double s = gvec[i];
      for (int j = i + 1; j < k; ++j) s -= H[(size_t)j * (m + 1) + i] * y[j];
      y[i] = s / H[(size_t)i * (m + 1) + i];
    }
    if (k > 0) {
      std::copy(y.begin(), y.begin() + k, ctx->scal_h + 512);
      NXFX_CUDA(ctx, cudaMemcpyAsync(ycoef, ctx->scal_h + 512, k * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
      if ((rc = do_multi_axpy(ctx, n, k, Z, ld, ycoef, 1.0, x))) return rc;
    }
  }
  info->iterations = its;
  info->converged = std::isfinite(info->residual_norm) && info->residual_norm <= tol;
  return NXFX_OK;
}

// row tiles of the pipelined SpMV (shared by the symbolic phase and the generic pattern upload)
int setup_spmv_tiles(nxfx_ctx* ctx) {
  const int n = (int)ctx->ndofs;
  const int ntiles = (int)cdiv(n, kTileRows);
  NXFX_CUDA(ctx, ctx->tile_base.alloc((size_t)ntiles + 2));
  int32_t* max_tile = reinterpret_cast<int32_t*>(ctx->ticket.p);  // borrowed, reset below
  NXFX_LAUNCH(ctx, tile_base_kernel, (int)cdiv(ntiles + 1, kThreads), kThreads, 0, n, ntiles, ctx->rowptr.p,
              ctx->tile_base.p, max_tile);
  int32_t max_tile_h = 0;
  NXFX_CUDA(ctx, cudaMemcpyAsync(&max_tile_h, max_tile, sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream));
  NXFX_CUDA(ctx, cudaMemsetAsync(ctx->ticket.p, 0, sizeof(unsigned int), ctx->stream));
  NXFX_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  // every tile, widened to 16-byte boundaries (up to 3 entries on each side), fits the ring at once
  ctx->pipe_ok = pipe_tile_bytes(kTileRows, max_tile_h + 6) <= kRingBytes;
  if (ctx->pipe_ok) {
    const void* modes[] = {reinterpret_cast<const void*>(spmv_pipe_kernel<0>), reinterpret_cast<const void*>(spmv_pipe_kernel<1>),
                           reinterpret_cast<const void*>(spmv_pipe_kernel<2>), reinterpret_cast<const void*>(spmv_pipe_kernel<3>)};
    for (const void* k : modes) {
      NXFX_CUDA(ctx, cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kPipeSmem));
      NXFX_CUDA(ctx, cudaFuncSetAttribute(k, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared));
    }
  }
  return NXFX_OK;
}

}  // namespace

// =============================================================================================
extern "C" {

int nxfx_abi_version(void) { return NXFX_ABI_VERSION; }

int nxfx_create(nxfx_ctx** out, int device) {
  if (!out) return NXFX_ERR_INVALID;
  *out = nullptr;
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || device < 0 || device >= count) return NXFX_ERR_CUDA;
  if (cudaSetDevice(device) != cudaSuccess) return NXFX_ERR_CUDA;
  auto* ctx = new nxfx_ctx();
  ctx->device = device;
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) == cudaSuccess) ctx->sm_count = prop.multiProcessorCount;
  cudaEventCreate(&ctx->ev0);
  cudaEventCreate(&ctx->ev1);
  *out = ctx;
  return NXFX_OK;
}

int nxfx_destroy(nxfx_ctx* ctx) {
  if (!ctx) return NXFX_OK;
  cudaSetDevice(ctx->device);
  cudaStreamSynchronize(ctx->stream);
  if (ctx->ev0) cudaEventDestroy(ctx->ev0);
  if (ctx->ev1) cudaEventDestroy(ctx->ev1);
  if (ctx->scal_h) cudaFreeHost(ctx->scal_h);
  if (ctx->side) cudaStreamDestroy(ctx->side);
  if (ctx->ev_x) cudaEventDestroy(ctx->ev_x);
  nxfx_comm_destroy(ctx);
  release_matrices(ctx);
  delete ctx;
  return NXFX_OK;
}

const char* nxfx_last_error(const nxfx_ctx* ctx) { return ctx ? ctx->err.c_str() : "null ctx"; }

int nxfx_set_stream(nxfx_ctx* ctx, void* s) {
  if (!ctx) return NXFX_ERR_INVALID;
  ctx->stream = reinterpret_cast<cudaStream_t>(s);
  return NXFX_OK;
}

int nxfx_sync(nxfx_ctx* ctx) {
  if (!ctx) return NXFX_ERR_INVALID;
  NXFX_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return NXFX_OK;
}

int64_t nxfx_launch_count(const nxfx_ctx* ctx) { return ctx ? ctx->launches : -1; }

int nxfx_malloc(nxfx_ctx* ctx, size_t bytes, void** out) {
  if (!ctx || !out) return NXFX_ERR_INVALID;
  NXFX_CUDA(ctx, cudaMalloc(out, bytes ? bytes : 8));
  return NXFX_OK;
}
int nxfx_free(nxfx_ctx* ctx, void* p) {
  if (!ctx) return NXFX_ERR_INVALID;
  NXFX_CUDA(ctx, cudaFree(p));
  return NXFX_OK;
}
int nxfx_host_alloc(nxfx_ctx* ctx, size_t bytes, void** out) {
  if (!ctx || !out) return NXFX_ERR_INVALID;
  NXFX_CUDA(ctx, cudaHostAlloc(out, bytes ? bytes : 8, cudaHostAllocDefault));
  return NXFX_OK;
}
int nxfx_host_free(nxfx_ctx* ctx, void* p) {
  if (!ctx) return NXFX_ERR_INVALID;
  NXFX_CUDA(ctx, cudaFreeHost(p));
  return NXFX_OK;
}
int nxfx_memcpy_h2d(nxfx_ctx* ctx, void* d, const void* s, size_t bytes) {
  if (!ctx) return NXFX_ERR_INVALID;
  NXFX_CUDA(ctx, cudaMemcpyAsync(d, s, bytes, cudaMemcpyHostToDevice, ctx->stream));
  return NXFX_OK;
}
int nxfx_memcpy_d2h(nxfx_ctx* ctx, void* d, const void* s, size_t bytes) {
  if (!ctx) return NXFX_ERR_INVALID;
  NXFX_CUDA(ctx, cudaMemcpyAsync(d, s, bytes, cudaMemcpyDeviceToHost, ctx->stream));
  return NXFX_OK;
}
int nxfx_memcpy_d2d(nxfx_ctx* ctx, void* d, const void* s, size_t bytes) {
  if (!ctx) return NXFX_ERR_INVALID;
  NXFX_CUDA(ctx, cudaMemcpyAsync(d, s, bytes, cudaMemcpyDeviceToDevice, ctx->stream));
  return NXFX_OK;
}
int nxfx_memset(nxfx_ctx* ctx, void* d, int byte, size_t bytes) {
  if (!ctx) return NXFX_ERR_INVALID;
  NXFX_CUDA(ctx, cudaMemsetAsync(d, byte, bytes, ctx->stream));
  return NXFX_OK;
}
int nxfx_timer_start(nxfx_ctx* ctx) {
  if (!ctx) return NXFX_ERR_INVALID;
  NXFX_CUDA(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
  return NXFX_OK;
}
int nxfx_timer_stop(nxfx_ctx* ctx, double* ms) {
  if (!ctx || !ms) return NXFX_ERR_INVALID;
  NXFX_CUDA(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
  NXFX_CUDA(ctx, cudaEventSynchronize(ctx->ev1));
  float f = 0.f;
  NXFX_CUDA(ctx, cudaEventElapsedTime(&f, ctx->ev0, ctx->ev1));
  *ms = f;
  return NXFX_OK;
}

// ---- (1) graph -> mesh -------------------------------------------------------------------------
int nxfx_set_network(nxfx_ctx* ctx, int32_t n_nodes, int32_t n_edges, int32_t gdim, int32_t N,
                     const double* node_pos, const int32_t* edge_u, const int32_t* edge_v,
                     const int32_t* edge_slot, const int32_t* node_lm, int32_t n_bif,
                     const int32_t* bif_ptr, const int32_t* bif_inc) {
  if (!ctx) return NXFX_ERR_INVALID;
  NXFX_REQUIRE(ctx, n_nodes > 0 && n_edges > 0 && N >= 1 && gdim >= 1 && gdim <= 3, "bad sizes");
  NXFX_REQUIRE(ctx, node_pos && edge_u && edge_v && edge_slot && node_lm && bif_ptr, "null input");
  NXFX_CUDA(ctx, cudaSetDevice(ctx->device));
  const int64_t E = n_edges;
  const int64_t nq = E * (N + 1), nc = E * N, ndofs = nq + nc + n_bif;
  const int64_t nv = (int64_t)n_nodes + E * (N - 1);
  NXFX_REQUIRE(ctx, ndofs < (int64_t)2147483000 && nv * 3 < (int64_t)2147483000, "network too large for int32 indexing");
  const int32_t n_inc = bif_ptr[n_bif];
  NXFX_REQUIRE(ctx, n_inc == 0 || bif_inc, "null incidence list");
  // host-side validation + slot tables
  std::vector<int4> uvl((size_t)E);
  std::vector<int32_t> slot_edge((size_t)E, -1);
  for (int64_t e = 0; e < E; ++e) {
    const int32_t u = edge_u[e], v = edge_v[e], s = edge_slot[e];
    if (u < 0 || u >= n_nodes || v < 0 || v >= n_nodes || u == v)
      return fail(ctx, NXFX_ERR_INVALID, "edge %lld has invalid endpoints (%d, %d)", (long long)e, u, v);
    if (s < 0 || s >= E || slot_edge[s] != -1)
      return fail(ctx, NXFX_ERR_INVALID, "edge_slot is not a permutation (edge %lld -> %d)", (long long)e, s);
    if (node_lm[u] >= n_bif || node_lm[v] >= n_bif)
      return fail(ctx, NXFX_ERR_INVALID, "node_lm out of range at edge %lld", (long long)e);
    slot_edge[s] = (int32_t)e;
    uvl[s] = make_int4(u, v, node_lm[u], node_lm[v]);
  }
  for (int32_t k = 0; k < n_inc; ++k)
    if ((bif_inc[k] >> 1) < 0 || (bif_inc[k] >> 1) >= E)
      return fail(ctx, NXFX_ERR_INVALID, "bif_inc[%d] out of range", k);
  ctx->has_network = ctx->has_pattern = ctx->has_pbc = ctx->pc_ready = false;
  release_matrices(ctx);
  nxfx_comm_destroy(ctx);
  ctx->edge_slot_h.assign(edge_slot, edge_slot + E);
  ctx->n_shared = 0;
  ctx->shared_lm.release();
  ctx->shared_lm_h.clear();
  ctx->top_sh_pos.release();
  ctx->top_sh_idx.release();
  ctx->tree.t_of_bif_h.clear();
  ctx->lam_weight.release();
  ctx->lam_nonshared.release();
  ctx->p_nonshared.release();
  ctx->tree.set = false;
  ctx->n_nodes = n_nodes; ctx->E = n_edges; ctx->gdim = gdim; ctx->N = N; ctx->n_bif = n_bif;
  ctx->n_inc = n_inc; ctx->nv = nv; ctx->nc = nc; ctx->nq = nq; ctx->poff = nq; ctx->loff = nq + nc;
  ctx->ndofs = ndofs; ctx->nnz = 0;
  int rc;
  if ((rc = upload(ctx, ctx->pos_stage, node_pos, (size_t)n_nodes * gdim))) return rc;
  if ((rc = upload(ctx, ctx->edge_u, edge_u, (size_t)E))) return rc;
  if ((rc = upload(ctx, ctx->edge_v, edge_v, (size_t)E))) return rc;
  if ((rc = upload(ctx, ctx->edge_slot, edge_slot, (size_t)E))) return rc;
  if ((rc = upload(ctx, ctx->slot_edge, slot_edge.data(), (size_t)E))) return rc;
  if ((rc = upload(ctx, ctx->slot_uvl, uvl.data(), (size_t)E))) return rc;
  std::vector<int2> uv((size_t)E);
  for (int64_t s = 0; s < E; ++s) uv[s] = make_int2(uvl[s].x, uvl[s].y);
  if ((rc = upload(ctx, ctx->slot_uv, uv.data(), (size_t)E))) return rc;
  std::vector<int2> lm((size_t)E);
  for (int64_t s = 0; s < E; ++s) lm[s] = make_int2(uvl[s].z, uvl[s].w);
  if ((rc = upload(ctx, ctx->slot_lm, lm.data(), (size_t)E))) return rc;
  std::vector<uint32_t> in_bits((size_t)(n_inc + 31) / 32 + 1, 0u);
  for (int32_t k = 0; k < n_inc; ++k)
    if (bif_inc[k] & 1) in_bits[k >> 5] |= 1u << (k & 31);
  if ((rc = upload(ctx, ctx->bif_in_bits, in_bits.data(), in_bits.size()))) return rc;
  DevBuf<int32_t> node_lm_d;
  if ((rc = upload(ctx, node_lm_d, node_lm, (size_t)n_nodes))) return rc;
  if ((rc = upload(ctx, ctx->bif_ptr, bif_ptr, (size_t)n_bif + 1))) return rc;
  if ((rc = upload(ctx, ctx->bif_inc, bif_inc, (size_t)n_inc))) return rc;
  NXFX_CUDA(ctx, ctx->x.alloc((size_t)nv * 4));
  NXFX_CUDA(ctx, cudaMemsetAsync(ctx->x.p, 0, (size_t)nv * 4 * sizeof(double), ctx->stream));
  NXFX_CUDA(ctx, ctx->edge_g.alloc((size_t)E));
  NXFX_CUDA(ctx, ctx->edge_c.alloc((size_t)E));
  NXFX_CUDA(ctx, ctx->edge_fn.alloc((size_t)E));
  if ((rc = ensure_scal(ctx))) return rc;
  if ((rc = build_vertices(ctx))) return rc;
  // bifurcation vertices carry their multiplier index in the (there unused) boundary-pressure slot
  NXFX_LAUNCH(ctx, tag_lm_kernel, (int)cdiv(n_nodes, kThreads), kThreads, 0, n_nodes, node_lm_d.p, ctx->x.p);
  NXFX_CUDA(ctx, cudaStreamSynchronize(ctx->stream));  // host vectors go out of scope
  ctx->has_network = true;
  return NXFX_OK;
}

int nxfx_update_node_positions(nxfx_ctx* ctx, const double* node_pos) {
  if (!ctx) return NXFX_ERR_INVALID;
  NXFX_REQUIRE(ctx, ctx->has_network && node_pos, "no network / null input");
  NXFX_CUDA(ctx, cudaMemcpyAsync(ctx->pos_stage.p, node_pos, (size_t)ctx->n_nodes * ctx->gdim * sizeof(double),
                                 cudaMemcpyHostToDevice, ctx->stream));
  return build_vertices(ctx);
}

int nxfx_get_sizes(const nxfx_ctx* ctx, int64_t* nv, int64_t* nc, int64_t* ndofs, int64_t* nnz) {
  if (!ctx || !ctx->has_network) return NXFX_ERR_INVALID;
  if (nv) *nv = ctx->nv;
  if (nc) *nc = ctx->nc;
  if (ndofs) *ndofs = ctx->ndofs;
  if (nnz) *nnz = ctx->nnz;
  return NXFX_OK;
}

int nxfx_mesh_geometry_device(nxfx_ctx* ctx, const double** x) {
  if (!ctx || !x) return NXFX_ERR_INVALID;
  NXFX_REQUIRE(ctx, ctx->has_network, "no network");
  *x = ctx->x.p;
  return NXFX_OK;
}

// ---- (2) symbolic --------------------------------------------------------------------------------
int nxfx_symbolic(nxfx_ctx* ctx) {
  if (!ctx) return NXFX_ERR_INVALID;
  NXFX_REQUIRE(ctx, ctx->has_network, "no network");
  int rc;
  ctx->generic = false;
  const int n = (int)ctx->ndofs;
  Net g = make_net(ctx);
  DevBuf<int32_t> len;
  NXFX_CUDA(ctx, len.alloc((size_t)n + 1));
  NXFX_CUDA(ctx, ctx->rowptr.alloc((size_t)n + 1 + 8));  // +8: bulk copies round sizes up to 16 B
  NXFX_CUDA(ctx, cudaMemsetAsync(ctx->rowptr.p, 0, ((size_t)n + 9) * sizeof(int32_t), ctx->stream));
  NXFX_LAUNCH(ctx, row_len_kernel, (int)cdiv(n + 1, kThreads), kThreads, 0, g, len.p);
  size_t tmp_bytes = 0;
  NXFX_CUDA(ctx, cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, len.p, ctx->rowptr.p, n + 1, ctx->stream));
  DevBuf<char> tmp;
  NXFX_CUDA(ctx, tmp.alloc(tmp_bytes));
  NXFX_CUDA(ctx, cub::DeviceScan::ExclusiveSum(tmp.p, tmp_bytes, len.p, ctx->rowptr.p, n + 1, ctx->stream));
  ctx->launches++;
  int32_t nnz = 0;
  NXFX_CUDA(ctx, cudaMemcpyAsync(&nnz, ctx->rowptr.p + n, sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream));
  NXFX_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  NXFX_REQUIRE(ctx, nnz > 0, "pattern overflow (nnz does not fit int32)");
  ctx->nnz = nnz;
  NXFX_CUDA(ctx, ctx->colidx.alloc((size_t)nnz + 8));
  NXFX_CUDA(ctx, cudaMemsetAsync(ctx->colidx.p, 0, ((size_t)nnz + 8) * sizeof(int32_t), ctx->stream));
  NXFX_LAUNCH(ctx, fill_cols_kernel, (int)cdiv(n, kThreads), kThreads, 0, g, ctx->rowptr.p, ctx->colidx.p);
  if ((rc = setup_spmv_tiles(ctx))) return rc;
  release_matrices(ctx);  // a new pattern: matrices of the previous one are gone (matrix 0 is created on demand)
  ctx->has_pattern = true;
  return NXFX_OK;
}

int nxfx_matrix_create(nxfx_ctx* ctx, int64_t* mat_id) {
  if (!ctx || !mat_id) return NXFX_ERR_INVALID;
  NXFX_REQUIRE(ctx, ctx->has_pattern, "symbolic phase has not been run");
  MatState* m = nullptr;
  int rc = new_matrix(ctx, ctx->next_mat_id++, &m);
  if (rc) return rc;
  *mat_id = m->id;
  return NXFX_OK;
}

static MatState* find_matrix(nxfx_ctx* ctx, int64_t id) {
  for (MatState* m : ctx->mats)
    if (m->id == id) return m;
  return nullptr;
}

int nxfx_matrix_destroy(nxfx_ctx* ctx, int64_t mat_id) {
  if (!ctx) return NXFX_ERR_INVALID;
  for (size_t i = 0; i < ctx->mats.size(); ++i) {
    if (ctx->mats[i]->id != mat_id) continue;
    NXFX_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (ctx->cur == ctx->mats[i]) { ctx->cur = nullptr; ctx->bottom_factored = false; }
    if (ctx->pc_mat == mat_id) { ctx->pc_ready = false; ctx->pc_mat = -1; }
    delete ctx->mats[i];
    ctx->mats.erase(ctx->mats.begin() + (long)i);
    return NXFX_OK;
  }
  return NXFX_OK;  // already gone with its pattern
}

int nxfx_matrix_bind(nxfx_ctx* ctx, int64_t mat_id) {
  if (!ctx) return NXFX_ERR_INVALID;
  MatState* m = find_matrix(ctx, mat_id);
  if (!m) return fail(ctx, NXFX_ERR_INVALID, "nxfx_matrix_bind: matrix %lld does not exist on the current pattern", (long long)mat_id);
  bind_matrix(ctx, m);
  return NXFX_OK;
}

int nxfx_matrix_zero(nxfx_ctx* ctx) {
  if (!ctx) return NXFX_ERR_INVALID;
  NXFX_REQUIRE(ctx, ctx->has_pattern, "symbolic phase has not been run");
  { int rc = ensure_matrix(ctx); if (rc) return rc; }
  MatState* m = ctx->cur;
  NXFX_CUDA(ctx, cudaMemsetAsync(m->vals.p, 0, m->vals.n * sizeof(double), ctx->stream));
  NXFX_CUDA(ctx, cudaMemsetAsync(m->cell_rh.p, 0, m->cell_rh.n * sizeof(double), ctx->stream));
  m->assembled = false;
  m->acc_count = 0;
  m->static_valid = false;
  if (ctx->pc_mat == m->id) ctx->pc_ready = false;
  return NXFX_OK;
}

int nxfx_matrix_touch(nxfx_ctx* ctx) {
  if (!ctx) return NXFX_ERR_INVALID;
  NXFX_REQUIRE(ctx, ctx->has_pattern, "symbolic phase has not been run");
  { int rc = ensure_matrix(ctx); if (rc) return rc; }
  ctx->cur->static_valid = false;
  return NXFX_OK;
}

int nxfx_matrix_static_valid(nxfx_ctx* ctx, int32_t* valid) {
  if (!ctx || !valid) return NXFX_ERR_INVALID;
  NXFX_REQUIRE(ctx, ctx->has_pattern, "symbolic phase has not been run");
  { int rc = ensure_matrix(ctx); if (rc) return rc; }
  *valid = ctx->cur->static_valid;
  return NXFX_OK;
}

int nxfx_matrix_info(nxfx_ctx* ctx, int64_t* mat_id, int32_t* assembled, int32_t* acc_count) {
  if (!ctx) return NXFX_ERR_INVALID;
  NXFX_REQUIRE(ctx, ctx->has_pattern, "symbolic phase has not been run");
  { int rc = ensure_matrix(ctx); if (rc) return rc; }
  if (mat_id) *mat_id = ctx->cur->id;
  if (assembled) *assembled = ctx->cur->assembled;
  if (acc_count) *acc_count = ctx->cur->acc_count;
  return NXFX_OK;
}

int nxfx_csr_device(nxfx_ctx* ctx, const int32_t** rowptr, const int32_t** colidx, double** vals) {
  if (!ctx) return NXFX_ERR_INVALID;
  NXFX_REQUIRE(ctx, ctx->has_pattern, "symbolic phase has not been run");
  { int rc = ensure_matrix(ctx); if (rc) return rc; }
  if (rowptr) *rowptr = ctx->rowptr.p;
  if (colidx) *colidx = ctx->colidx.p;
  if (vals) *vals = ctx->cur->vals.p;
  return NXFX_OK;
}

// ---- (3) numeric ---------------------------------------------------------------------------------
int nxfx_set_boundary_pressure(nxfx_ctx* ctx, const double* pbc) {
  if (!ctx || !pbc) return NXFX_ERR_INVALID;
  NXFX_REQUIRE(ctx, ctx->has_network, "no network");
  NXFX_LAUNCH(ctx, set_pbc_kernel, (int)cdiv(ctx->nv, kThreads), kThreads, 0, ctx->nv, pbc, ctx->x.p);
  ctx->has_pbc = true;
  return NXFX_OK;
}

int nxfx_assemble(nxfx_ctx* ctx, const double* R_cell, double R_const, const double* f_cell,
                  double f_const, int lhs, int rhs, int accumulate, double* b) {
  if (!ctx) return NXFX_ERR_INVALID;
  NXFX_REQUIRE(ctx, ctx->has_pattern, "symbolic phase has not been run");
  NXFX_REQUIRE(ctx, !ctx->generic, "higher-order pattern loaded: use nxfx_assemble_generic");
  NXFX_REQUIRE(ctx, !rhs || (b && ctx->has_pbc), "rhs requested without b / boundary pressure");
  NXFX_REQUIRE(ctx, !rhs || (reinterpret_cast<uintptr_t>(b) & 15) == 0, "b must be 16-byte aligned");
  if (!lhs && !rhs) return NXFX_OK;
  { int rc = ensure_matrix(ctx); if (rc) return rc; }
  Net g = make_net(ctx);
  Coef c;
  c.R_cell = R_cell; c.f_cell = f_cell; c.R_const = R_const; c.f_const = f_const;
  c.cell_rh = ctx->cur->cell_rh.p;
  const bool n1 = ctx->N == 1;
  const int nft = (int)cdiv(ctx->nq, n1 ? kFluxRowsN1 : kTileRows);
  const int npt = (int)cdiv(ctx->nc, kPresRows);
  const int nlt = (int)cdiv(ctx->n_bif, kLamRows);
  const int grid = nft + npt + nlt;
  // a re-assembly that overwrites leaves the pressure / multiplier rows (pattern-only values) in place
  const int ws = !(lhs && !accumulate && ctx->cur->static_valid);
  if (accumulate) {
    if (n1) NXFX_LAUNCH(ctx, (assemble_tiles_kernel<true, true>), grid, kTileRows, 0, g, c, ctx->rowptr.p, ctx->cur->vals.p, b, lhs, rhs, ws, nft, npt);
    else NXFX_LAUNCH(ctx, (assemble_tiles_kernel<true, false>), grid, kTileRows, 0, g, c, ctx->rowptr.p, ctx->cur->vals.p, b, lhs, rhs, ws, nft, npt);
  } else {
    if (n1) NXFX_LAUNCH(ctx, (assemble_tiles_kernel<false, true>), grid, kTileRows, 0, g, c, ctx->rowptr.p, ctx->cur->vals.p, b, lhs, rhs, ws, nft, npt);
    else NXFX_LAUNCH(ctx, (assemble_tiles_kernel<false, false>), grid, kTileRows, 0, g, c, ctx->rowptr.p, ctx->cur->vals.p, b, lhs, rhs, ws, nft, npt);
  }
  if (lhs) {
    note_lhs_assembled(ctx, accumulate);
    ctx->cur->static_valid = !accumulate;  // ADD_VALUES turns them into k * {-1, +1}, k * (0, +-1)
  }
  return NXFX_OK;
}

// ---- (4) solve -----------------------------------------------------------------------------------
int nxfx_set_tree_schedule(nxfx_ctx* ctx, const int32_t* t_of_bif, const int32_t* t_parent,
                           const int32_t* t_pedge, const int32_t* t_cptr, const int32_t* t_cidx,
                           int32_t n_chunks, const int32_t* chunk_lptr, int32_t n_lvl_ptr,
                           const int32_t* lvl_ptr, int32_t n_chords, const int32_t* chord_edge) {
  if (!ctx) return NXFX_ERR_INVALID;
  NXFX_REQUIRE(ctx, ctx->has_network, "no network");
  auto& s = ctx->tree;
  s.set = false;
  const size_t nb = (size_t)ctx->n_bif;
  if (nb == 0) { s.n_chunks = 0; s.set = true; return NXFX_OK; }
  NXFX_REQUIRE(ctx, t_of_bif && t_parent && t_pedge && t_cptr && chunk_lptr && lvl_ptr && n_chunks >= 1, "null input");
  NXFX_REQUIRE(ctx, chunk_lptr[0] == 0 && chunk_lptr[n_chunks] == n_lvl_ptr - 1 && lvl_ptr[0] == 0 &&
                        lvl_ptr[n_lvl_ptr - 1] == ctx->n_bif, "inconsistent level tables");
  for (size_t t = 0; t < nb; ++t) {
    // (a parent without a local link edge is legal: multi-GPU, the link belongs to another rank)
    if (t_parent[t] >= (int32_t)nb || t_pedge[t] >= ctx->E || (t_pedge[t] >= 0 && t_parent[t] < 0))
      return fail(ctx, NXFX_ERR_INVALID, "tree schedule: bad parent at %zu", t);
  }
  int rc;
  if ((rc = upload(ctx, s.t_of_bif, t_of_bif, nb))) return rc;
  std::vector<int32_t> inv(nb);
  for (size_t i = 0; i < nb; ++i) {
    if (t_of_bif[i] < 0 || (size_t)t_of_bif[i] >= nb) return fail(ctx, NXFX_ERR_INVALID, "t_of_bif out of range");
    inv[t_of_bif[i]] = (int32_t)i;
  }
  if ((rc = upload(ctx, s.bif_of_t, inv.data(), nb))) return rc;
  NXFX_CUDA(ctx, s.lam_nat.alloc(nb));
  {  // incidences of every node in schedule order (read by the fused N == 1 tree kernels)
    DevBuf<int32_t> len;
    NXFX_CUDA(ctx, len.alloc(nb + 1));
    NXFX_CUDA(ctx, s.t_inc_ptr.alloc(nb + 1));
    NXFX_CUDA(ctx, s.t_inc.alloc((size_t)std::max(ctx->n_inc, 1)));
    NXFX_LAUNCH(ctx, t_inc_len_kernel, (int)cdiv(nb + 1, kThreads), kThreads, 0, (int)nb, s.bif_of_t.p, ctx->bif_ptr.p, len.p);
    size_t tmp_bytes = 0;
    NXFX_CUDA(ctx, cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, len.p, s.t_inc_ptr.p, (int)nb + 1, ctx->stream));
    DevBuf<char> tmp;
    NXFX_CUDA(ctx, tmp.alloc(tmp_bytes));
    NXFX_CUDA(ctx, cub::DeviceScan::ExclusiveSum(tmp.p, tmp_bytes, len.p, s.t_inc_ptr.p, (int)nb + 1, ctx->stream));
    NXFX_LAUNCH(ctx, t_inc_fill_kernel, (int)cdiv(nb, kThreads), kThreads, 0, (int)nb, s.bif_of_t.p, ctx->bif_ptr.p,
                ctx->bif_inc.p, ctx->edge_slot.p, s.t_inc_ptr.p, s.t_inc.p);
    NXFX_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  }
  if ((rc = upload(ctx, s.t_parent, t_parent, nb))) return rc;
  if ((rc = upload(ctx, s.t_pedge, t_pedge, nb))) return rc;
  {
    std::vector<int32_t> pslot(nb);
    for (size_t t = 0; t < nb; ++t) pslot[t] = t_pedge[t] >= 0 ? ctx->edge_slot_h[t_pedge[t]] : -1;
    if ((rc = upload(ctx, s.t_pslot, pslot.data(), nb))) return rc;
    NXFX_CUDA(ctx, cudaStreamSynchronize(ctx->stream));  // pslot goes out of scope
  }
  if ((rc = upload(ctx, s.t_cptr, t_cptr, nb + 1))) return rc;
  if ((rc = upload(ctx, s.t_cidx, t_cidx, (size_t)t_cptr[nb]))) return rc;
  if ((rc = upload(ctx, s.chunk_lptr, chunk_lptr, (size_t)n_chunks + 1))) return rc;
  if ((rc = upload(ctx, s.lvl_ptr, lvl_ptr, (size_t)n_lvl_ptr))) return rc;
  if ((rc = upload(ctx, s.chord_edge, chord_edge, (size_t)std::max(0, n_chords)))) return rc;
  s.n_chunks = n_chunks; s.n_lvl_ptr = n_lvl_ptr; s.n_chords = n_chords;
  s.n_top = lvl_ptr[chunk_lptr[n_chunks]] - lvl_ptr[chunk_lptr[n_chunks - 1]];
  s.top_b0 = lvl_ptr[chunk_lptr[n_chunks - 1]];
  s.t_of_bif_h.assign(t_of_bif, t_of_bif + nb);
  s.top_lvl_h.assign(lvl_ptr + chunk_lptr[n_chunks - 1], lvl_ptr + chunk_lptr[n_chunks] + 1);
  // shared-memory sweeps need every chunk (nodes, levels) to fit the on-chip tables
  s.fast_ok = true;
  int max_nodes = 0, max_links = 0;
  for (int c = 0; c < n_chunks; ++c) {
    const int l0 = chunk_lptr[c], l1 = chunk_lptr[c + 1];
    if (l1 - l0 > kLevelCap) s.fast_ok = false;
    max_nodes = std::max(max_nodes, lvl_ptr[l1] - lvl_ptr[l0]);
    max_links = std::max(max_links, t_cptr[lvl_ptr[l1]] - t_cptr[lvl_ptr[l0]]);
  }
  s.cap = (max_nodes <= 2048 && max_links <= 4096) ? 2048 : kChunkCapMax;
  if (max_nodes > s.cap || max_links > 2 * s.cap) s.fast_ok = false;
  if (s.fast_ok) {
    std::vector<int32_t> desc((size_t)n_chunks * kDescInts, 0);
    for (int c = 0; c < n_chunks; ++c) {
      int32_t* d = desc.data() + (size_t)c * kDescInts;
      const int l0 = chunk_lptr[c], l1 = chunk_lptr[c + 1];
      d[0] = lvl_ptr[l0]; d[1] = lvl_ptr[l1]; d[2] = t_cptr[d[0]]; d[3] = t_cptr[d[1]]; d[4] = l1 - l0;
      int lw = -1;  // levels 0..lw have <= 32 nodes: handled by one warp
      while (lw + 1 < l1 - l0 && lvl_ptr[l0 + lw + 2] - lvl_ptr[l0 + lw + 1] <= 32) ++lw;
      d[5] = lw;
      for (int l = l0; l <= l1; ++l) d[8 + l - l0] = lvl_ptr[l];
    }
    if ((rc = upload(ctx, s.chunk_desc, desc.data(), desc.size()))) return rc;
    NXFX_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    // single-launch solve: needs every bottom chunk resident at once
    s.coop_ok = false;
    int coop = 0, per_sm = 0;
    cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, ctx->device);
    if (coop && cudaFuncSetAttribute(tree_solve_coop_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     (int)tree_smem_bytes(kChunkCapMax)) == cudaSuccess &&
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, tree_solve_coop_kernel, kTreeThreads, tree_smem_bytes(ctx->tree.cap)) == cudaSuccess)
      s.coop_ok = n_chunks <= per_sm * ctx->sm_count;  // bottom blocks + one block for the top chunk
    cudaGetLastError();
    NXFX_CUDA(ctx, cudaFuncSetAttribute(tree_factor_solve_bottom_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tree_smem_bytes_fs(kChunkCapMax)));
    NXFX_CUDA(ctx, cudaFuncSetAttribute((tree_top_split_kernel<FactorSolveOp, kPartial>), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tree_smem_bytes_fs(kChunkCapMax)));
    NXFX_CUDA(ctx, cudaFuncSetAttribute((tree_top_split_kernel<FactorSolveOp, kFinish>), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tree_smem_bytes_fs(kChunkCapMax)));
    s.coop_fs_ok = false;
    per_sm = 0;
    const int fs_max = (int)tree_smem_bytes_fs(kChunkCapMax);
    if (coop &&
        cudaFuncSetAttribute(tree_factor_solve_coop_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, fs_max) == cudaSuccess &&
        cudaFuncSetAttribute(tree_factor_solve_coop_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, fs_max) == cudaSuccess &&
        cudaFuncSetAttribute(tree_factor_solve_coop_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, fs_max) == cudaSuccess &&
        cudaFuncSetAttribute(tree_factor_solve_coop_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, fs_max) == cudaSuccess &&
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, tree_factor_solve_coop_kernel<true, true>, kTreeThreads,
                                                      tree_smem_bytes_fs(ctx->tree.cap)) == cudaSuccess) {
      // bottom blocks + one block for the top chunk; with more chunks than that, several chunks per block
      s.coop_fs_blocks = per_sm * ctx->sm_count;
      s.coop_fs_ok = s.coop_fs_blocks >= 2;
    }
    cudaGetLastError();
    NXFX_CUDA(ctx, cudaFuncSetAttribute(tree_factor_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tree_smem_bytes(kChunkCapMax)));
    NXFX_CUDA(ctx, cudaFuncSetAttribute((tree_top_split_kernel<FactorOp, kPartial>), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tree_smem_bytes(kChunkCapMax)));
    NXFX_CUDA(ctx, cudaFuncSetAttribute((tree_top_split_kernel<FactorOp, kFinish>), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tree_smem_bytes(kChunkCapMax)));
    NXFX_CUDA(ctx, cudaFuncSetAttribute((tree_top_split_kernel<SolveOp, kPartial>), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tree_smem_bytes(kChunkCapMax)));
    NXFX_CUDA(ctx, cudaFuncSetAttribute((tree_top_split_kernel<SolveOp, kFinish>), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tree_smem_bytes(kChunkCapMax)));
    NXFX_CUDA(ctx, cudaFuncSetAttribute(tree_solve_kernel<kTreeUp>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tree_smem_bytes(kChunkCapMax)));
    NXFX_CUDA(ctx, cudaFuncSetAttribute(tree_solve_kernel<kTreeDown>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tree_smem_bytes(kChunkCapMax)));
  }
  NXFX_CUDA(ctx, s.tg.alloc(nb));
  NXFX_CUDA(ctx, s.diag0.alloc(nb));
  NXFX_CUDA(ctx, s.d.alloc(nb));
  NXFX_CUDA(ctx, s.gd.alloc(nb));
  NXFX_CUDA(ctx, s.r.alloc(nb));
  NXFX_CUDA(ctx, s.lam.alloc(nb));
  NXFX_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  s.set = true;
  ctx->pc_ready = false;
  return update_top_shared(ctx);
}

int nxfx_pc_setup(nxfx_ctx* ctx) {
  if (!ctx) return NXFX_ERR_INVALID;
  return do_pc_setup(ctx);
}

int nxfx_pc_apply(nxfx_ctx* ctx, const double* r, double* z) {
  if (!ctx || !r || !z) return NXFX_ERR_INVALID;
  return do_pc_apply(ctx, NXFX_PC_NETWORK_SCHUR, r, z);
}

int nxfx_spmv(nxfx_ctx* ctx, const double* x, double* y) {
  if (!ctx || !x || !y) return NXFX_ERR_INVALID;
  NXFX_REQUIRE(ctx, ctx->has_pattern, "symbolic phase has not been run");
  { int rc = ensure_matrix(ctx); if (rc) return rc; }
  return do_spmv(ctx, x, y);
}

int nxfx_residual(nxfx_ctx* ctx, const double* b, const double* x, double* r, double* norm2) {
  if (!ctx || !b || !x || !r) return NXFX_ERR_INVALID;
  NXFX_REQUIRE(ctx, ctx->has_pattern, "symbolic phase has not been run");
  int rc = ensure_matrix(ctx);
  if (rc) return rc;
  rc = do_residual(ctx, b, x, r, slot(ctx, 0));
  if (rc) return rc;
  if (norm2) {
    NXFX_CUDA(ctx, cudaMemcpyAsync(ctx->scal_h, slot(ctx, 0), sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    NXFX_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    *norm2 = ctx->scal_h[0];
  }
  return NXFX_OK;
}

int nxfx_solve(nxfx_ctx* ctx, const double* b, double* x, const nxfx_solve_opts* opts, nxfx_solve_info* info) {
  if (!ctx || !b || !x || !opts || !info) return NXFX_ERR_INVALID;
  NXFX_REQUIRE(ctx, is_assembled(ctx), "matrix has not been assembled");
  std::memset(info, 0, sizeof *info);
  int rc;
  if (opts->pc_type == NXFX_PC_NETWORK_SCHUR && ctx->generic && !ctx->cond.set)
    return fail(ctx, NXFX_ERR_UNSUPPORTED, "higher-order elements: call nxfx_set_condensation before a direct solve");
  bool fused_setup = false;
  if (ctx->comm.ready)
    NXFX_REQUIRE(ctx, can_fuse_setup(ctx) || (ctx->pc_ready && ctx->cur->acc_count == 1),
                 "the fused partitioned solve needs a forest schedule that fits the cooperative kernel");
  if (opts->pc_type == NXFX_PC_NETWORK_SCHUR && !ctx->pc_ready) {
    // a fresh matrix and a direct solve: factorise while eliminating the right-hand side
    fused_setup = opts->ksp_type == NXFX_KSP_PREONLY && can_fuse_setup(ctx);
    if (!fused_setup && (rc = do_pc_setup(ctx))) return rc;
  }
  if (ctx->comm.ready)
    NXFX_REQUIRE(ctx, opts->ksp_type == NXFX_KSP_PREONLY && opts->pc_type == NXFX_PC_NETWORK_SCHUR,
                 "the partitioned solve is the direct one (ksp_type preonly, pc_type lu)");
  if (opts->ksp_type == NXFX_KSP_PREONLY) rc = solve_preonly(ctx, b, x, opts, info, fused_setup);
  else if (opts->ksp_type == NXFX_KSP_FGMRES) rc = solve_fgmres(ctx, b, x, opts, info);
  else return fail(ctx, NXFX_ERR_UNSUPPORTED, "unknown ksp_type %d", opts->ksp_type);
  if (rc) return rc;
  if (ctx->mirror_h) {
    if (opts->ksp_type != NXFX_KSP_PREONLY && (rc = mirror_copy(ctx, x))) return rc;
    NXFX_CUDA(ctx, cudaStreamSynchronize(ctx->side));
  }
  if (ctx->comm.ready && *ctx->comm.err_h) {
    *ctx->comm.err_h = 0;
    return fail(ctx, NXFX_ERR_COMM, "a peer rank did not deliver its part of the exchange within 4 s");
  }
  if (!info->converged && opts->error_if_not_converged)
    return fail(ctx, NXFX_ERR_NOT_CONVERGED, "linear solve did not converge: ||r|| = %.3e, ||b|| = %.3e after %d iterations",
                info->residual_norm, info->rhs_norm, info->iterations);
  return NXFX_OK;
}

int nxfx_set_solution_mirror(nxfx_ctx* ctx, double* x_h) {
  if (!ctx) return NXFX_ERR_INVALID;
  if (x_h && !ctx->side) {
    NXFX_CUDA(ctx, cudaStreamCreateWithFlags(&ctx->side, cudaStreamNonBlocking));
    NXFX_CUDA(ctx, cudaEventCreateWithFlags(&ctx->ev_x, cudaEventDisableTiming));
  }
  ctx->mirror_h = x_h;
  return NXFX_OK;
}

// ---- (5) end-to-end host-buffer step ---------------------------------------------------------------
int nxfx_assemble_solve_host(nxfx_ctx* ctx, const double* node_pos, const double* pbc_vertex,
                             double R_const, double f_const, const nxfx_solve_opts* opts, double* x_h,
                             nxfx_solve_info* info) {
  if (!ctx || !node_pos || !pbc_vertex || !opts || !x_h || !info) return NXFX_ERR_INVALID;
  NXFX_REQUIRE(ctx, ctx->has_pattern, "symbolic phase has not been run");
  const size_t n = (size_t)ctx->ndofs;
  if (ctx->e2e_b.n < n) {
    NXFX_CUDA(ctx, ctx->e2e_b.alloc(n));
    NXFX_CUDA(ctx, ctx->e2e_x.alloc(n));
    NXFX_CUDA(ctx, ctx->e2e_pbc.alloc((size_t)ctx->nv));
  }
  int rc;
  if ((rc = nxfx_update_node_positions(ctx, node_pos))) return rc;
  NXFX_CUDA(ctx, cudaMemcpyAsync(ctx->e2e_pbc.p, pbc_vertex, (size_t)ctx->nv * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
  if ((rc = nxfx_set_boundary_pressure(ctx, ctx->e2e_pbc.p))) return rc;
  if ((rc = nxfx_assemble(ctx, nullptr, R_const, nullptr, f_const, 1, 1, 0, ctx->e2e_b.p))) return rc;
  if ((rc = nxfx_solve(ctx, ctx->e2e_b.p, ctx->e2e_x.p, opts, info))) return rc;
  NXFX_CUDA(ctx, cudaMemcpyAsync(x_h, ctx->e2e_x.p, n * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
  NXFX_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return NXFX_OK;
}

// ---- (7) table-driven assembly for higher-order elements ------------------------------------------
int nxfx_set_generic_system(nxfx_ctx* ctx, int32_t n_dofs, int32_t n_flux_rows, int32_t nnz,
                            const int32_t* rowptr, const int32_t* colidx, const int32_t* src_id,
                            const double* src_coef, const int32_t* bsrc_ptr, const int32_t* bsrc_id,
                            const double* bsrc_coef) {
  if (!ctx) return NXFX_ERR_INVALID;
  NXFX_REQUIRE(ctx, ctx->has_network, "no network");
  NXFX_REQUIRE(ctx, n_dofs > 0 && nnz > 0 && n_flux_rows >= 0 && n_flux_rows <= n_dofs, "bad sizes");
  NXFX_REQUIRE(ctx, rowptr && colidx && src_id && src_coef && bsrc_ptr, "null input");
  NXFX_REQUIRE(ctx, rowptr[0] == 0 && rowptr[n_dofs] == nnz, "rowptr does not match nnz");
  const int64_t nc = ctx->nc;
  for (int64_t k = 0; k < 2 * (int64_t)nnz; ++k) {
    const int32_t s = src_id[k];
    if (s >= 0 && (s & (kRhFlag - 1)) >= nc) return fail(ctx, NXFX_ERR_INVALID, "src_id[%lld] out of range", (long long)k);
  }
  for (int32_t k = 0; k < nnz; ++k)
    if (colidx[k] < 0 || colidx[k] >= n_dofs) return fail(ctx, NXFX_ERR_INVALID, "colidx[%d] out of range", k);
  const int32_t nb = bsrc_ptr[n_dofs];
  for (int32_t k = 0; k < nb; ++k) {
    const int32_t i = bsrc_id[k];
    const int64_t lim = (i & kVertexFlag) ? ctx->nv : nc;
    if (i < 0 || (i & (kVertexFlag - 1)) >= lim) return fail(ctx, NXFX_ERR_INVALID, "bsrc_id[%d] out of range", k);
  }
  int rc;
  ctx->has_pattern = ctx->pc_ready = false;
  ctx->cond.set = false;
  release_matrices(ctx);
  ctx->ndofs = n_dofs; ctx->nq = n_flux_rows; ctx->nnz = nnz;
  ctx->poff = n_flux_rows; ctx->loff = n_dofs - ctx->n_bif;
  NXFX_CUDA(ctx, ctx->rowptr.alloc((size_t)n_dofs + 9));
  NXFX_CUDA(ctx, cudaMemsetAsync(ctx->rowptr.p, 0, ((size_t)n_dofs + 9) * sizeof(int32_t), ctx->stream));
  NXFX_CUDA(ctx, cudaMemcpyAsync(ctx->rowptr.p, rowptr, ((size_t)n_dofs + 1) * sizeof(int32_t), cudaMemcpyHostToDevice, ctx->stream));
  NXFX_CUDA(ctx, ctx->colidx.alloc((size_t)nnz + 8));
  NXFX_CUDA(ctx, cudaMemsetAsync(ctx->colidx.p, 0, ((size_t)nnz + 8) * sizeof(int32_t), ctx->stream));
  NXFX_CUDA(ctx, cudaMemcpyAsync(ctx->colidx.p, colidx, (size_t)nnz * sizeof(int32_t), cudaMemcpyHostToDevice, ctx->stream));
  if ((rc = upload(ctx, ctx->gen_src_id, src_id, (size_t)2 * nnz))) return rc;
  if ((rc = upload(ctx, ctx->gen_src_coef, src_coef, (size_t)2 * nnz))) return rc;
  if ((rc = upload(ctx, ctx->gen_bptr, bsrc_ptr, (size_t)n_dofs + 1))) return rc;
  if ((rc = upload(ctx, ctx->gen_bid, bsrc_id, (size_t)nb))) return rc;
  if ((rc = upload(ctx, ctx->gen_bcoef, bsrc_coef, (size_t)nb))) return rc;
  NXFX_CUDA(ctx, ctx->gen_cell_h.alloc((size_t)nc));
  if ((rc = setup_spmv_tiles(ctx))) return rc;
  ctx->generic = true;
  ctx->has_pattern = true;
  return NXFX_OK;
}

int nxfx_assemble_generic(nxfx_ctx* ctx, const double* R_cell, double R_const, const double* f_cell,
                          double f_const, int lhs, int rhs, int accumulate, double* b) {
  if (!ctx) return NXFX_ERR_INVALID;
  NXFX_REQUIRE(ctx, ctx->has_pattern && ctx->generic, "nxfx_set_generic_system has not been called");
  NXFX_REQUIRE(ctx, !rhs || (b && ctx->has_pbc), "rhs requested without b / boundary pressure");
  if (!lhs && !rhs) return NXFX_OK;
  { int rc = ensure_matrix(ctx); if (rc) return rc; }
  Net g = make_net(ctx);
  NXFX_LAUNCH(ctx, cell_length_kernel, vec_grid(ctx, ctx->nc), kThreads, 0, g, ctx->gen_cell_h.p);
  if (lhs) {
    const int2* sid = reinterpret_cast<const int2*>(ctx->gen_src_id.p);
    const double2* sco = reinterpret_cast<const double2*>(ctx->gen_src_coef.p);
    if (accumulate)
      NXFX_LAUNCH(ctx, assemble_generic_kernel<true>, vec_grid(ctx, ctx->nnz), kThreads, 0, ctx->nnz, sid, sco,
                  ctx->gen_cell_h.p, R_cell, R_const, ctx->cur->vals.p);
    else
      NXFX_LAUNCH(ctx, assemble_generic_kernel<false>, vec_grid(ctx, ctx->nnz), kThreads, 0, ctx->nnz, sid, sco,
                  ctx->gen_cell_h.p, R_cell, R_const, ctx->cur->vals.p);
    // R*h per cell travels with the values (the condensation is built from it), accumulated like them
    if (accumulate && ctx->cur->assembled)
      NXFX_LAUNCH(ctx, cell_rh_generic_kernel<true>, vec_grid(ctx, ctx->nc), kThreads, 0, ctx->nc, ctx->gen_cell_h.p, R_cell,
                  R_const, ctx->cur->cell_rh.p);
    else
      NXFX_LAUNCH(ctx, cell_rh_generic_kernel<false>, vec_grid(ctx, ctx->nc), kThreads, 0, ctx->nc, ctx->gen_cell_h.p, R_cell,
                  R_const, ctx->cur->cell_rh.p);
    note_lhs_assembled(ctx, accumulate);
  }
  if (rhs) {
    const int n = (int)ctx->ndofs;
    if (accumulate)
      NXFX_LAUNCH(ctx, rhs_generic_kernel<true>, (int)cdiv(n, kThreads), kThreads, 0, n, ctx->gen_bptr.p, ctx->gen_bid.p,
                  ctx->gen_bcoef.p, ctx->gen_cell_h.p, f_cell, f_const, g.x2, b);
    else
      NXFX_LAUNCH(ctx, rhs_generic_kernel<false>, (int)cdiv(n, kThreads), kThreads, 0, n, ctx->gen_bptr.p, ctx->gen_bid.p,
                  ctx->gen_bcoef.p, ctx->gen_cell_h.p, f_cell, f_const, g.x2, b);
  }
  return NXFX_OK;
}

int nxfx_set_condensation(nxfx_ctx* ctx, int32_t continuous_pressure, int32_t flux_dofs_per_edge, int32_t n_max,
                          int32_t kl, int32_t pcell_base, int32_t pcell_stride, const int32_t* type_n,
                          const int32_t* loc_ptr, const int32_t* loc_kind, const int32_t* loc_off,
                          const int32_t* k_ptr, const int32_t* k_row, const int32_t* k_col, const int32_t* k_cell,
                          const double* k_coef, const int32_t* c_ptr, const int32_t* c_row, const int32_t* c_slot,
                          const double* c_coef, const int32_t* d_ptr, const int32_t* d_slot, const int32_t* d_col,
                          const double* d_coef, const int32_t* bif_node) {
  if (!ctx) return NXFX_ERR_INVALID;
  NXFX_REQUIRE(ctx, ctx->has_pattern && ctx->generic, "nxfx_set_generic_system has not been called");
  NXFX_REQUIRE(ctx, type_n && loc_ptr && loc_kind && loc_off && k_ptr && k_row && k_col && k_cell && k_coef && c_ptr &&
                        d_ptr && (ctx->n_bif == 0 || bif_node), "null input");
  NXFX_REQUIRE(ctx, n_max > 0 && kl > 0 && flux_dofs_per_edge > 0 && pcell_base >= 0 && pcell_stride >= 0, "bad sizes");
  auto& k = ctx->cond;
  k.set = false;
  ctx->pc_ready = false;
  const int64_t E = ctx->E, nd = ctx->ndofs;
  for (int t = 0; t < 4; ++t) {
    const int n = type_n[t];
    if (n <= 0 || n > n_max || loc_ptr[t + 1] - loc_ptr[t] != n) return fail(ctx, NXFX_ERR_INVALID, "condensation: bad type_n[%d]", t);
    for (int i = loc_ptr[t]; i < loc_ptr[t + 1]; ++i) {
      // the largest global index any edge can produce for this local unknown must be a dof
      int64_t top;
      switch (loc_kind[i]) {
        case 0: top = (E - 1) * flux_dofs_per_edge + loc_off[i]; break;
        case 1: top = pcell_base + (E - 1) * (int64_t)pcell_stride + loc_off[i]; break;
        case 2: top = ctx->nq + ctx->n_nodes + (E - 1) * (int64_t)(ctx->N - 1) + loc_off[i]; break;
        case 3: case 4: top = ctx->nq + ctx->n_nodes - 1; break;
        default: return fail(ctx, NXFX_ERR_INVALID, "condensation: unknown kind %d", loc_kind[i]);
      }
      if (loc_off[i] < 0 || top >= nd) return fail(ctx, NXFX_ERR_INVALID, "condensation: local unknown %d out of range", i);
    }
    for (int i = k_ptr[t]; i < k_ptr[t + 1]; ++i)
      if (k_row[i] < 0 || k_row[i] >= n || k_col[i] < 0 || k_col[i] >= n || std::abs(k_row[i] - k_col[i]) > kl ||
          k_cell[i] >= ctx->N)
        return fail(ctx, NXFX_ERR_INVALID, "condensation: K entry %d out of range", i);
    for (int i = c_ptr[t]; i < c_ptr[t + 1]; ++i)
      if (c_row[i] < 0 || c_row[i] >= n || c_slot[i] < 0 || c_slot[i] > 3) return fail(ctx, NXFX_ERR_INVALID, "condensation: C entry %d out of range", i);
    for (int i = d_ptr[t]; i < d_ptr[t + 1]; ++i)
      if (d_col[i] < 0 || d_col[i] >= n || d_slot[i] < 0 || d_slot[i] > 3) return fail(ctx, NXFX_ERR_INVALID, "condensation: D entry %d out of range", i);
  }
  for (int32_t b = 0; b < ctx->n_bif; ++b)
    if (bif_node[b] < 0 || bif_node[b] >= ctx->n_nodes) return fail(ctx, NXFX_ERR_INVALID, "condensation: bif_node[%d] out of range", b);
  int rc;
  if ((rc = upload(ctx, k.type_n, type_n, 4))) return rc;
  if ((rc = upload(ctx, k.loc_ptr, loc_ptr, 5))) return rc;
  if ((rc = upload(ctx, k.loc_kind, loc_kind, (size_t)loc_ptr[4]))) return rc;
  if ((rc = upload(ctx, k.loc_off, loc_off, (size_t)loc_ptr[4]))) return rc;
  if ((rc = upload(ctx, k.k_ptr, k_ptr, 5))) return rc;
  if ((rc = upload(ctx, k.k_row, k_row, (size_t)k_ptr[4]))) return rc;
  if ((rc = upload(ctx, k.k_col, k_col, (size_t)k_ptr[4]))) return rc;
  if ((rc = upload(ctx, k.k_cell, k_cell, (size_t)k_ptr[4]))) return rc;
  if ((rc = upload(ctx, k.k_coef, k_coef, (size_t)k_ptr[4]))) return rc;
  if ((rc = upload(ctx, k.c_ptr, c_ptr, 5))) return rc;
  if ((rc = upload(ctx, k.c_row, c_row, (size_t)c_ptr[4]))) return rc;
  if ((rc = upload(ctx, k.c_slot, c_slot, (size_t)c_ptr[4]))) return rc;
  if ((rc = upload(ctx, k.c_coef, c_coef, (size_t)c_ptr[4]))) return rc;
  if ((rc = upload(ctx, k.d_ptr, d_ptr, 5))) return rc;
  if ((rc = upload(ctx, k.d_slot, d_slot, (size_t)d_ptr[4]))) return rc;
  if ((rc = upload(ctx, k.d_col, d_col, (size_t)d_ptr[4]))) return rc;
  if ((rc = upload(ctx, k.d_coef, d_coef, (size_t)d_ptr[4]))) return rc;
  if ((rc = upload(ctx, k.bif_node, bif_node, (size_t)ctx->n_bif))) return rc;
  NXFX_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  k.n_max = n_max; k.kl = kl; k.per_edge = flux_dofs_per_edge; k.pcell_base = pcell_base; k.pcell_stride = pcell_stride;
  k.cont = continuous_pressure ? 1 : 0;
  k.bif_node_h.assign(bif_node, bif_node + ctx->n_bif);
  NXFX_CUDA(ctx, cudaFuncSetAttribute(cond_edge_rhs_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kCondSmemMax));
  NXFX_CUDA(ctx, cudaFuncSetAttribute(cond_factor_group_kernel<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kCondSmemMax));
  NXFX_CUDA(ctx, cudaFuncSetAttribute(cond_factor_group_kernel<16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kCondSmemMax));
  NXFX_CUDA(ctx, cudaFuncSetAttribute(cond_factor_group_kernel<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kCondSmemMax));
  const size_t Es = (size_t)E, nb = (size_t)std::max(ctx->n_bif, 1);
  NXFX_CUDA(ctx, k.band.alloc((size_t)(3 * kl + 1) * n_max * Es));
  NXFX_CUDA(ctx, k.ipiv.alloc((size_t)n_max * Es));
  NXFX_CUDA(ctx, k.Y.alloc((size_t)4 * n_max * Es));
  NXFX_CUDA(ctx, k.S.alloc(16 * Es));
  NXFX_CUDA(ctx, k.y0.alloc((size_t)n_max * Es));
  NXFX_CUDA(ctx, k.h.alloc(4 * Es));
  for (auto* buf : {&k.bd0, &k.bU, &k.bL, &k.bDinv, &k.bG, &k.bH}) NXFX_CUDA(ctx, buf->alloc(4 * nb));
  NXFX_CUDA(ctx, k.br.alloc(2 * nb));
  NXFX_CUDA(ctx, k.bz.alloc(2 * nb));
  k.set = true;
  return update_pressure_weight(ctx);
}

// ---- (6) multi-GPU: partitioned network ----------------------------------------------------------
int nxfx_set_shared(nxfx_ctx* ctx, int32_t n_shared, const int32_t* shared_lm, const double* lam_weight) {
  if (!ctx) return NXFX_ERR_INVALID;
  NXFX_REQUIRE(ctx, ctx->has_network, "no network");
  NXFX_REQUIRE(ctx, n_shared >= 0 && n_shared <= ctx->n_bif && (n_shared == 0 || shared_lm) && lam_weight, "bad arguments");
  for (int32_t i = 0; i < n_shared; ++i)
    if (shared_lm[i] < 0 || shared_lm[i] >= ctx->n_bif) return fail(ctx, NXFX_ERR_INVALID, "shared_lm[%d] out of range", i);
  int rc;
  if ((rc = upload(ctx, ctx->shared_lm, shared_lm, (size_t)n_shared))) return rc;
  if ((rc = upload(ctx, ctx->lam_weight, lam_weight, (size_t)ctx->n_bif))) return rc;
  std::vector<double> nonshared((size_t)ctx->n_bif);
  for (int32_t i = 0; i < ctx->n_bif; ++i) nonshared[i] = lam_weight[i];
  for (int32_t i = 0; i < n_shared; ++i) nonshared[shared_lm[i]] = 0.0;
  if ((rc = upload(ctx, ctx->lam_nonshared, nonshared.data(), (size_t)ctx->n_bif))) return rc;
  NXFX_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  ctx->n_shared = n_shared;
  ctx->shared_lm_h.assign(shared_lm, shared_lm + n_shared);
  if ((rc = update_pressure_weight(ctx))) return rc;
  return update_top_shared(ctx);
}

static int dist_ready(nxfx_ctx* ctx, const double* buf) {
  // (the block sweeps of the table-driven path run out of global memory: any schedule fits them)
  NXFX_REQUIRE(ctx, ctx->tree.set && (ctx->tree.fast_ok || ctx->generic) && ctx->tree.n_chunks >= 1 && buf,
               "needs a tree schedule that fits the shared-memory sweeps and a buffer");
  NXFX_REQUIRE(ctx, !ctx->generic || ctx->cond.set, "nxfx_set_condensation has not been called");
  NXFX_REQUIRE(ctx, ctx->cur && ctx->cur->acc_count <= 1,
               "the partitioned solve does not take a matrix accumulated over several assemblies");
  NXFX_REQUIRE(ctx, ctx->n_shared == 0 || ctx->top_sh_pos.p, "nxfx_set_shared / nxfx_set_tree_schedule have not both been called");
  return NXFX_OK;
}

// doubles of the three exchanged sections (see nxfx_exchange_sizes)
static void exchange_sizes(const nxfx_ctx* ctx, int32_t* setup, int32_t* apply, int32_t* residual) {
  const int32_t nt = std::max(ctx->n_shared, 1);
  const bool cont = ctx->generic && ctx->cond.cont;
  *setup = (ctx->generic ? 12 : 2) * nt;
  *apply = (ctx->generic ? 2 : 1) * nt;
  *residual = (cont ? 3 : 1) * ctx->n_shared + 2;
}

int nxfx_exchange_sizes(nxfx_ctx* ctx, int32_t* setup, int32_t* apply, int32_t* residual) {
  if (!ctx || !setup || !apply || !residual) return NXFX_ERR_INVALID;
  NXFX_REQUIRE(ctx, ctx->tree.set && ctx->tree.n_chunks >= 1, "no tree schedule");
  NXFX_REQUIRE(ctx, !ctx->generic || ctx->cond.set, "nxfx_set_condensation has not been called");
  exchange_sizes(ctx, setup, apply, residual);
  return NXFX_OK;
}

int nxfx_pc_setup_begin(nxfx_ctx* ctx, double* buf) {
  if (!ctx) return NXFX_ERR_INVALID;
  int rc = dist_ready(ctx, buf);
  if (rc) return rc;
  NXFX_REQUIRE(ctx, is_assembled(ctx), "assemble the matrix before pc_setup");
  if ((rc = factor_bottom(ctx)) || (rc = top_split<true, kPartial>(ctx, buf))) return rc;
  ctx->bottom_factored = true;
  return NXFX_OK;
}

int nxfx_pc_setup_end(nxfx_ctx* ctx, double* buf) {
  if (!ctx) return NXFX_ERR_INVALID;
  int rc = dist_ready(ctx, buf);
  if (rc) return rc;
  NXFX_REQUIRE(ctx, ctx->bottom_factored, "nxfx_pc_setup_begin has not been run");
  if ((rc = top_split<true, kFinish>(ctx, buf))) return rc;
  mark_factored(ctx);
  return NXFX_OK;
}

int nxfx_pc_apply_begin(nxfx_ctx* ctx, const double* r, double* buf) {
  if (!ctx || !r) return NXFX_ERR_INVALID;
  int rc = dist_ready(ctx, buf);
  if (rc) return rc;
  // the forward sweep of the bottom chunks only needs THEIR factors: it may run before
  // nxfx_pc_setup_end, so that setup and first application share one all-reduce
  NXFX_REQUIRE(ctx, ctx->pc_ready || ctx->bottom_factored, "nxfx_pc_setup_begin has not been run");
  if ((rc = check_aligned(ctx, r)) || (rc = forward_bottom(ctx, r))) return rc;
  return top_split<false, kPartial>(ctx, buf);
}

int nxfx_pc_apply_end(nxfx_ctx* ctx, const double* r, double* z, double* buf, int add) {
  if (!ctx || !r || !z) return NXFX_ERR_INVALID;
  int rc = dist_ready(ctx, buf);
  if (rc) return rc;
  NXFX_REQUIRE(ctx, ctx->pc_ready, "pc_setup has not been run");
  if ((rc = top_split<false, kFinish>(ctx, buf))) return rc;
  return backward_bottom(ctx, r, z, add != 0);
}

// setup + first application in one pair of calls around ONE all-reduce of [setup | apply] sections.
// P1/DG0, N == 1: the bottom chunks are factorised while their right-hand sides are eliminated (one kernel),
// the top chunk handles factor and solve together in each phase; otherwise the four separate phases.
int nxfx_pc_setup_apply_begin(nxfx_ctx* ctx, const double* r, double* buf) {
  if (!ctx || !r) return NXFX_ERR_INVALID;
  int rc = dist_ready(ctx, buf);
  if (rc) return rc;
  NXFX_REQUIRE(ctx, is_assembled(ctx), "assemble the matrix before pc_setup");
  if (!fused_split(ctx)) {
    int32_t ns, na, nr;
    exchange_sizes(ctx, &ns, &na, &nr);
    if ((rc = nxfx_pc_setup_begin(ctx, buf))) return rc;
    return nxfx_pc_apply_begin(ctx, r, buf + ns);
  }
  if ((rc = check_aligned(ctx, r))) return rc;
  auto& s = ctx->tree;
  TreeDev t = make_tree(ctx);
  const int nb = s.n_chunks - 1;
  FusedN1 fin{make_net(ctx), r, ctx->cur->cell_rh.p, ctx->lam_weight.p};
  const size_t smem = tree_smem_bytes_fs(s.cap);
  if (nb > 0) NXFX_LAUNCH(ctx, tree_factor_solve_bottom_kernel, nb, kTreeThreads, smem, t, fin);
  NXFX_LAUNCH(ctx, (tree_top_split_kernel<FactorSolveOp, kPartial>), 1, kTreeThreads, smem, t, nb, buf, fin);
  ctx->bottom_factored = true;
  return NXFX_OK;
}

int nxfx_pc_setup_apply_end(nxfx_ctx* ctx, const double* r, double* z, double* buf) {
  if (!ctx || !r || !z) return NXFX_ERR_INVALID;
  int rc = dist_ready(ctx, buf);
  if (rc) return rc;
  if (!fused_split(ctx)) {
    int32_t ns, na, nr;
    exchange_sizes(ctx, &ns, &na, &nr);
    if ((rc = nxfx_pc_setup_end(ctx, buf))) return rc;
    return nxfx_pc_apply_end(ctx, r, z, buf + ns, 0);
  }
  NXFX_REQUIRE(ctx, ctx->bottom_factored, "nxfx_pc_setup_apply_begin has not been run");
  FusedN1 fin{make_net(ctx), r, ctx->cur->cell_rh.p, ctx->lam_weight.p};
  NXFX_LAUNCH(ctx, (tree_top_split_kernel<FactorSolveOp, kFinish>), 1, kTreeThreads, tree_smem_bytes_fs(ctx->tree.cap), make_tree(ctx),
              ctx->tree.n_chunks - 1, buf, fin);
  mark_factored(ctx);
  return backward_bottom(ctx, r, z, false);
}

// ---- peer exchange over NVLink (peer.cuh) ----------------------------------------------------------
static size_t comm_bytes(const PeerComm& c) {
  return kPeerHeaderBytes + (size_t)kPeerChannels * 2 * (size_t)c.nranks * (size_t)c.slot * sizeof(double);
}

int nxfx_comm_destroy(nxfx_ctx* ctx) {
  if (!ctx) return NXFX_ERR_INVALID;
  PeerComm& c = ctx->comm;
  if (!c.created) return NXFX_OK;
  cudaStreamSynchronize(ctx->stream);
  for (int r = 0; r < c.nranks; ++r)
    if (r != c.rank && c.base[r] && !c.in_process) cudaIpcCloseMemHandle(c.base[r]);
  if (c.local) cudaFree(c.local);
  if (c.err_h) cudaFreeHost(c.err_h);
  c.lam_scratch.release();
  c = PeerComm();
  cudaGetLastError();
  return NXFX_OK;
}

int nxfx_comm_create(nxfx_ctx* ctx, int32_t rank, int32_t nranks, void* handle_out, int32_t* slot_doubles) {
  if (!ctx || !handle_out) return NXFX_ERR_INVALID;
  if (ctx->generic)
    return fail(ctx, NXFX_ERR_UNSUPPORTED, "the in-kernel exchange is implemented for flux degree 1 / pressure degree 0 "
                "only; use the split phases (nxfx_pc_*_begin/_end) instead");
  NXFX_REQUIRE(ctx, nranks >= 2 && nranks <= kMaxPeers && rank >= 0 && rank < nranks, "bad rank / nranks");
  NXFX_REQUIRE(ctx, ctx->tree.set && ctx->lam_nonshared.p, "call nxfx_set_tree_schedule and nxfx_set_shared first");
  // the exchange lives in the fused cooperative tree kernel: one cell per edge, all chunks of this rank co-resident
  if (!(ctx->tree.fast_ok && ctx->tree.coop_fs_ok && ctx->tree.n_chunks > 1 && ctx->pipe_ok))
    return fail(ctx, NXFX_ERR_UNSUPPORTED, "the in-kernel exchange needs a schedule whose %d chunks fit the cooperative tree "
                "kernel at once; use the split phases (nxfx_pc_*_begin/_end) instead", ctx->tree.n_chunks);
  static_assert(sizeof(cudaIpcMemHandle_t) == NXFX_COMM_HANDLE_BYTES, "handle size");
  nxfx_comm_destroy(ctx);
  PeerComm& c = ctx->comm;
  c.rank = rank;
  c.nranks = nranks;
  c.slot = 2 * ((3 * std::max(ctx->n_shared, 1) + 1) & ~1);  // 3 n_shared values (>= n_shared + 2), two 8-byte words each
  NXFX_CUDA(ctx, cudaMalloc(&c.local, comm_bytes(c)));
  NXFX_CUDA(ctx, cudaMemset(c.local, 0, comm_bytes(c)));
  NXFX_CUDA(ctx, cudaHostAlloc(reinterpret_cast<void**>(&c.err_h), sizeof(int), cudaHostAllocMapped));
  *c.err_h = 0;
  NXFX_CUDA(ctx, cudaHostGetDevicePointer(reinterpret_cast<void**>(&c.err_d), c.err_h, 0));
  NXFX_CUDA(ctx, c.lam_scratch.alloc((size_t)std::max(ctx->n_bif, 1)));
  NXFX_CUDA(ctx, cudaDeviceSynchronize());
  cudaIpcMemHandle_t h;
  NXFX_CUDA(ctx, cudaIpcGetMemHandle(&h, c.local));
  std::memcpy(handle_out, &h, sizeof h);
  if (slot_doubles) *slot_doubles = c.slot;
  c.created = true;
  return NXFX_OK;
}

int nxfx_comm_connect(nxfx_ctx* ctx, const void* handles_all) {
  if (!ctx || !handles_all) return NXFX_ERR_INVALID;
  PeerComm& c = ctx->comm;
  NXFX_REQUIRE(ctx, c.created && !c.ready, "nxfx_comm_create has not been called (or the communicator is already connected)");
  const char* hs = static_cast<const char*>(handles_all);
  for (int r = 0; r < c.nranks; ++r) {
    if (r == c.rank) { c.base[r] = c.local; continue; }
    cudaIpcMemHandle_t h;
    std::memcpy(&h, hs + (size_t)r * sizeof h, sizeof h);
    cudaError_t e = cudaIpcOpenMemHandle(&c.base[r], h, cudaIpcMemLazyEnablePeerAccess);
    if (e != cudaSuccess) {
      cudaGetLastError();
      c.base[r] = nullptr;
      return fail(ctx, NXFX_ERR_COMM, "cudaIpcOpenMemHandle(rank %d) -> %s", r, cudaGetErrorString(e));
    }
  }
  c.ready = true;
  return NXFX_OK;
}

// peer access from ctx's device to `device` (idempotent; NXFX_ERR_COMM if the devices cannot reach each other)
static int enable_peer(nxfx_ctx* ctx, int device) {
  if (device == ctx->device || (device < 64 && (ctx->peer_on >> device) & 1u)) return NXFX_OK;
  int can = 0;
  NXFX_CUDA(ctx, cudaDeviceCanAccessPeer(&can, ctx->device, device));
  if (!can) return fail(ctx, NXFX_ERR_COMM, "device %d cannot access the memory of device %d (no peer access)", ctx->device, device);
  NXFX_CUDA(ctx, cudaSetDevice(ctx->device));
  const cudaError_t e = cudaDeviceEnablePeerAccess(device, 0);
  if (e == cudaErrorPeerAccessAlreadyEnabled) cudaGetLastError();
  else NXFX_CUDA(ctx, e);
  if (device < 64) ctx->peer_on |= 1ull << device;
  return NXFX_OK;
}

int nxfx_comm_connect_local(nxfx_ctx* ctx, nxfx_ctx* const* ctxs, int32_t nranks) {
  if (!ctx || !ctxs) return NXFX_ERR_INVALID;
  PeerComm& c = ctx->comm;
  NXFX_REQUIRE(ctx, c.created && !c.ready, "nxfx_comm_create has not been called (or the communicator is already connected)");
  NXFX_REQUIRE(ctx, nranks == c.nranks && ctxs[c.rank] == ctx, "nranks or this context's rank disagree with nxfx_comm_create");
  for (int r = 0; r < nranks; ++r) {
    const nxfx_ctx* o = ctxs[r];
    if (!o || !o->comm.created || o->comm.rank != r || o->comm.nranks != nranks || o->comm.slot != c.slot)
      return fail(ctx, NXFX_ERR_INVALID, "nxfx_comm_connect_local: context %d is not rank %d of the same %d-rank group "
                  "(nxfx_comm_create with the same nranks and slot size on every context)", r, r, nranks);
  }
  unsigned int flags = 0;
  NXFX_CUDA(ctx, cudaStreamGetFlags(ctx->stream, &flags));
  NXFX_REQUIRE(ctx, flags & cudaStreamNonBlocking,
               "in-process ranks need a stream created with cudaStreamNonBlocking (the legacy stream serialises them)");
  // Ranks on one device wait for each other inside the cooperative tree kernel: the grids of all of them must be
  // resident together, or a waiting grid holds the SMs its peer needs.  Same calculation as the single-rank check
  // (blocks per SM x SMs, tree.coop_fs_blocks), summed over the ranks of each device; every rank checks every
  // device, so all ranks reach the same verdict.
  bool shared = false;
  for (int r = 0; r < nranks; ++r) {
    int sum = 0, cap = INT32_MAX, k = 0;
    char list[160] = "";
    for (int q = 0; q < nranks; ++q) {
      if (ctxs[q]->device != ctxs[r]->device) continue;
      if (q < r) { k = -1; break; }  // device counted at its first rank
      const TreeSchedule& s = ctxs[q]->tree;
      const int grid = std::min(s.n_chunks - 1, s.coop_fs_blocks - 1) + 1;  // as do_pc_setup_apply launches it
      sum += grid;
      cap = std::min(cap, s.coop_fs_blocks);
      const size_t len = std::strlen(list);
      if (len + 16 < sizeof list) std::snprintf(list + len, sizeof list - len, "%s%d", k ? " + " : "", grid);
      ++k;
    }
    if (k < 2) continue;
    if (ctxs[r]->device == ctx->device) shared = true;
    if (sum > cap)
      return fail(ctx, NXFX_ERR_UNSUPPORTED, "the cooperative tree grids of the %d ranks on device %d are not resident together: "
                  "%s = %d blocks > %d (blocks per SM x SMs); use the split phases (nxfx_pc_*_begin/_end) instead",
                  k, ctxs[r]->device, list, sum, cap);
  }
  for (int r = 0; r < nranks; ++r) {
    int rc = enable_peer(ctx, ctxs[r]->device);
    if (rc) return rc;
  }
  // Everything the step needs from the driver happens now, not while a peer's kernel waits: the solve workspace is
  // allocated, and every kernel the step can launch is loaded (with lazy module loading, the first launch of a
  // kernel loads it under a lock that stalls the other ranks' threads -- measured on a B200: a peer's cooperative
  // grid was never launched and the exchange timed out)
  int rc = ensure_work(ctx, 3);
  if (rc) return rc;
  const void* step_kernels[] = {
      reinterpret_cast<const void*>(tree_factor_solve_coop_kernel<true, false>),
      reinterpret_cast<const void*>(tree_factor_solve_coop_kernel<true, true>),
      reinterpret_cast<const void*>(edge_backsub_n1_kernel<false>), reinterpret_cast<const void*>(edge_backsub_n1_kernel<true>),
      reinterpret_cast<const void*>(edge_backsub_kernel<false>), reinterpret_cast<const void*>(edge_backsub_kernel<true>),
      reinterpret_cast<const void*>(edge_condense_kernel<true>), reinterpret_cast<const void*>(bif_rhs_kernel<true>),
      reinterpret_cast<const void*>(spmv_pipe_kernel<3>)};
  for (const void* k : step_kernels) {
    cudaFuncAttributes fa;
    NXFX_CUDA(ctx, cudaFuncGetAttributes(&fa, k));
  }
  for (int r = 0; r < nranks; ++r) c.base[r] = ctxs[r]->comm.local;
  c.in_process = true;
  c.shared_device = shared;
  c.ready = true;
  return NXFX_OK;
}

int nxfx_group_sum(nxfx_ctx* ctx, const double* const* src, int32_t nranks, double* dst, int64_t n) {
  if (!ctx || !src || !dst || n < 0) return NXFX_ERR_INVALID;
  NXFX_REQUIRE(ctx, nranks >= 1 && nranks <= kMaxPeers, "nranks out of range");
  GroupSrc g = {};
  for (int r = 0; r < nranks; ++r) {
    NXFX_REQUIRE(ctx, src[r], "null source buffer");
    g.p[r] = src[r];
    cudaPointerAttributes a;
    NXFX_CUDA(ctx, cudaPointerGetAttributes(&a, src[r]));
    NXFX_REQUIRE(ctx, a.type == cudaMemoryTypeDevice, "sources must be device memory");
    int rc = enable_peer(ctx, a.device);
    if (rc) return rc;
  }
  if (n == 0) return NXFX_OK;
  NXFX_LAUNCH(ctx, group_sum_kernel, (int)std::min<int64_t>(cdiv(n, kGroupSumThreads), (int64_t)ctx->sm_count * 4),
              kGroupSumThreads, 0, g, (int)nranks, dst, n);
  return NXFX_OK;
}

int nxfx_residual_partial(nxfx_ctx* ctx, const double* b, const double* x, double* r, double* buf) {
  if (!ctx || !b || !x || !r || !buf) return NXFX_ERR_INVALID;
  NXFX_REQUIRE(ctx, ctx->has_pattern && ctx->lam_nonshared.p, "nxfx_set_shared has not been called");
  NXFX_REQUIRE(ctx, is_assembled(ctx), "matrix has not been assembled");
  NXFX_REQUIRE(ctx, !ctx->generic || ctx->cond.set, "nxfx_set_condensation has not been called");
  if (!ctx->generic && ctx->pipe_ok) {  // the weighted partial norms come out of the residual kernel itself
    const PipeShape ps = pipe_shape(ctx);
    NXFX_LAUNCH(ctx, spmv_pipe_kernel<2>, ps.grid, kPipeThreads, kPipeSmem, (int)ctx->ndofs, ps.ntiles, ctx->rowptr.p,
                ctx->colidx.p, ctx->cur->vals.p, ctx->tile_base.p, x, r, b, ctx->scal.p, ctx->ticket.p,
                buf + ctx->n_shared, (int)ctx->loff, ctx->lam_nonshared.p, ctx->lam_weight.p);
    return pack_shared(ctx, r, b, buf, false);
  }
  // [lam rows of r | (cont) P rows of r | (cont) P rows of b | norm partials without any shared row]: a plain
  // residual, then the packs and a weighted-norm kernel that also skips the nodal pressure rows of the shared
  // bifurcations
  const bool cont = ctx->generic && ctx->cond.cont && ctx->n_shared > 0;
  int rc;
  if ((rc = do_residual(ctx, b, x, r, slot(ctx, 0))) || (rc = pack_shared(ctx, r, b, buf, cont))) return rc;
  const int n = (int)ctx->ndofs, nr = (cont ? 3 : 1) * ctx->n_shared;
  NXFX_LAUNCH(ctx, weighted_norm2_pair_kernel, vec_grid(ctx, n), kThreads, 0, n, (int)ctx->loff, r, ctx->lam_nonshared.p,
              b, ctx->lam_weight.p, ctx->scal.p, ctx->ticket.p, buf + nr, (int)ctx->nq, cont ? ctx->n_nodes : 0,
              cont ? ctx->p_nonshared.p : nullptr);
  return NXFX_OK;
}

int nxfx_residual_finish(nxfx_ctx* ctx, const double* buf, double* r, double* nrm_out) {
  if (!ctx || !buf || !r || !nrm_out) return NXFX_ERR_INVALID;
  NXFX_REQUIRE(ctx, ctx->lam_nonshared.p, "nxfx_set_shared has not been called");
  if (ctx->generic) {
    NXFX_REQUIRE(ctx, ctx->cond.set, "nxfx_set_condensation has not been called");
    NXFX_LAUNCH(ctx, cond_residual_finish_kernel, 1, kThreads, 0, ctx->n_shared, (int)ctx->loff, (int)ctx->nq,
                ctx->cond.cont && ctx->n_shared > 0 ? 1 : 0, ctx->shared_lm.p, ctx->cond.bif_node.p, ctx->lam_weight.p,
                buf, r, nrm_out);
    return NXFX_OK;
  }
  NXFX_LAUNCH(ctx, residual_finish_kernel, 1, kThreads, 0, ctx->n_shared, (int)ctx->loff, ctx->shared_lm.p, buf, r, nrm_out);
  return NXFX_OK;
}

int nxfx_global_flux(nxfx_ctx* ctx, const double* x, double* out) {
  if (!ctx || !x || !out) return NXFX_ERR_INVALID;
  NXFX_REQUIRE(ctx, ctx->has_network, "no network");
  NXFX_LAUNCH(ctx, global_flux_kernel, vec_grid(ctx, ctx->nc), kThreads, 0, make_net(ctx), x, out);
  return NXFX_OK;
}

int nxfx_gather(nxfx_ctx* ctx, const double* src, const int32_t* map, int32_t S, int64_t n_rows, int32_t N,
                double* dst) {
  if (!ctx) return NXFX_ERR_INVALID;
  NXFX_REQUIRE(ctx, N >= 1 && (S == 1 || S == N) && n_rows >= 0, "N >= 1, S in {1, N}, n_rows >= 0");
  if (n_rows == 0) return NXFX_OK;
  NXFX_REQUIRE(ctx, src && dst, "null src / dst");
  NXFX_LAUNCH(ctx, gather_kernel, vec_grid(ctx, n_rows * N), kThreads, 0, n_rows, (int)N, (int)S, map, src, dst);
  return NXFX_OK;
}

#ifdef NXFX_TREE_STAMPS
// development builds only (not part of include/nxfx_b200.h)
int nxfx_debug_tree_stamps(nxfx_ctx* ctx, unsigned long long* out32) {
  if (!ctx || !out32) return NXFX_ERR_INVALID;
  NXFX_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  NXFX_CUDA(ctx, cudaMemcpyFromSymbol(out32, g_tree_stamps, 32 * sizeof(unsigned long long)));
  return NXFX_OK;
}
int nxfx_debug_device_attrs(nxfx_ctx* ctx, int* out8) {
  if (!ctx || !out8) return NXFX_ERR_INVALID;
  cudaDeviceGetAttribute(out8 + 0, cudaDevAttrL2CacheSize, ctx->device);
  cudaDeviceGetAttribute(out8 + 1, cudaDevAttrMaxPersistingL2CacheSize, ctx->device);
  cudaDeviceGetAttribute(out8 + 2, cudaDevAttrMaxAccessPolicyWindowSize, ctx->device);
  cudaDeviceGetAttribute(out8 + 3, cudaDevAttrMaxSharedMemoryPerMultiprocessor, ctx->device);
  cudaDeviceGetAttribute(out8 + 4, cudaDevAttrMultiProcessorCount, ctx->device);
  cudaDeviceGetAttribute(out8 + 5, cudaDevAttrCanUseHostPointerForRegisteredMem, ctx->device);
  cudaDeviceGetAttribute(out8 + 6, cudaDevAttrClusterLaunch, ctx->device);
  cudaDeviceGetAttribute(out8 + 7, cudaDevAttrMemoryPoolsSupported, ctx->device);
  return NXFX_OK;
}
#endif

}  // extern "C"
