// CSR SpMV and fused vector kernels for the Krylov solve (solver.py:127 replaces KSPSolve).
//
// A block owns tiles of kTileRows consecutive rows: the tile's (value, column) pairs are streamed
// from HBM, x is gathered from L2 (x is 8*n_dofs bytes, far below the 126 MB L2), the products are
// parked in shared memory and every row is reduced sequentially in ascending column order.  The
// row sum is therefore deterministic and bit-identical to a sequential CSR product (mul then add,
// no FMA).  MODE 1 fuses r = b - A x with the block partials of ||r||^2 and ||b||^2.
//   spmv_pipe_kernel  persistent blocks, TMA bulk copies (cp.async.bulk) + mbarrier pipeline,
//                     L2 evict-first hint on the matrix stream -- the production kernel;
//   spmv_kernel       plain loads, any tile size -- fallback for very long rows.
#pragma once

#include "ctx.cuh"
#include "peer.cuh"

namespace nxfx {

constexpr int kEntriesPerThread = kTileCap / kTileRows;  // 8
constexpr int kMaxPartials = 4096;

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
  return v;
}

// Block-wide sum (fixed tree => deterministic); result valid in thread 0.
template <int THREADS>
__device__ __forceinline__ double block_sum(double v, double* red /* [THREADS/32] */) {
  v = warp_sum(v);
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  if (lane == 0) red[w] = v;
  __syncthreads();
  double s = 0.0;
  if (w == 0) {
    s = lane < THREADS / 32 ? red[lane] : 0.0;
    s = warp_sum(s);
  }
  __syncthreads();
  return s;
}

// Last-block-done final reduction of per-block partials -> out[0..K).  Deterministic: the last
// block (whichever it is) sums the partials in index order with the same fixed tree.
template <int THREADS, int K>
__device__ __forceinline__ bool finish_partials(double (&mine)[K], double* partial, int nblocks,
                                                unsigned int* ticket, double* out, double* red) {
  __shared__ bool last;
  if (threadIdx.x == 0) {
#pragma unroll
    for (int k = 0; k < K; ++k) partial[(size_t)k * kMaxPartials + blockIdx.x] = mine[k];
    __threadfence();
    const unsigned int t = atomicAdd(ticket, 1u);
    last = (t == (unsigned int)nblocks - 1);
  }
  __syncthreads();
  if (!last) return false;
  __threadfence();
#pragma unroll
  for (int k = 0; k < K; ++k) {
    double s = 0.0;
    for (int i = threadIdx.x; i < nblocks; i += THREADS)
      s += ((volatile double*)partial)[(size_t)k * kMaxPartials + i];
    s = block_sum<THREADS>(s, red);
    if (threadIdx.x == 0) out[k] = s;
  }
  if (threadIdx.x == 0) *ticket = 0u;
  return true;
}

// MODE 0: y = A x.   MODE 1: y = b - A x and norm2_out[0] = ||y||^2, norm2_out[1] = ||b||^2
// MODE 2 (pipeline kernel): as 1 with the rows >= loff weighted by w_r / w_b (multi-GPU partial norms)
// MODE 3 (pipeline kernel): as 2, and the block that finishes last exchanges the shared multiplier rows
//         of r and the two norm partials with the other ranks over NVLink (peer_allgather), adds them up
//         in rank order, writes the reduced rows back into y and the GLOBAL norms to norm2_out
// (block partials, grid-strided tiles so that the partial count stays bounded).
template <int MODE>
__global__ void __launch_bounds__(kTileRows)
spmv_kernel(int n, int ntiles, const int32_t* __restrict__ rowptr,
            const int32_t* __restrict__ colidx, const double* __restrict__ vals,
            const double* __restrict__ x, double* __restrict__ y, const double* __restrict__ b,
            double* partial, unsigned int* ticket, double* norm2_out) {
  __shared__ double sm[kTileCap];
  __shared__ int srow[kTileRows + 1];
  __shared__ double red[kTileRows / 32];
  double nrm = 0.0, nrb = 0.0;
  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int r0 = tile * kTileRows;
    const int nr = min(kTileRows, n - r0);
    if (threadIdx.x <= nr) srow[threadIdx.x] = rowptr[r0 + threadIdx.x];
    if (threadIdx.x == 0) srow[nr] = rowptr[r0 + nr];
    __syncthreads();
    const int sbase = srow[0];
    const int tnnz = srow[nr] - sbase;
    const bool valid = threadIdx.x < nr;
    const int rs = valid ? srow[threadIdx.x] - sbase : 0;
    const int re = valid ? srow[threadIdx.x + 1] - sbase : 0;
    double acc = 0.0;
    for (int c0 = 0; c0 < tnnz; c0 += kTileCap) {
      const int cnt = min(kTileCap, tnnz - c0);
      const size_t g0 = (size_t)sbase + c0;
      double v[kEntriesPerThread];
      int c[kEntriesPerThread];
#pragma unroll
      for (int k = 0; k < kEntriesPerThread; ++k) {
        const int idx = threadIdx.x + k * kTileRows;
        if (idx < cnt) {
          v[k] = __ldg(vals + g0 + idx);
          c[k] = __ldg(colidx + g0 + idx);
        }
      }
#pragma unroll
      for (int k = 0; k < kEntriesPerThread; ++k) {
        const int idx = threadIdx.x + k * kTileRows;
        if (idx < cnt) sm[idx] = __dmul_rn(v[k], x[c[k]]);
      }
      __syncthreads();
      const int s = max(rs - c0, 0), e = min(re - c0, cnt);
      for (int k = s; k < e; ++k) acc = __dadd_rn(acc, sm[k]);
      __syncthreads();
    }
    if (valid) {
      if (MODE == 0) {
        y[r0 + threadIdx.x] = acc;
      } else {
        const double bi = b[r0 + threadIdx.x];
        const double r = __dsub_rn(bi, acc);
        y[r0 + threadIdx.x] = r;
        nrm += r * r;
        nrb += bi * bi;
      }
    }
  }
  if (MODE == 1) {
    double mine[2] = {block_sum<kTileRows>(nrm, red), block_sum<kTileRows>(nrb, red)};
    finish_partials<kTileRows, 2>(mine, partial, gridDim.x, ticket, norm2_out, red);
  }
}

// ---- pipelined SpMV (TMA bulk copies + mbarrier) -----------------------------------------------
// Persistent blocks walk over row tiles; thread 0 keeps kStages-1 tiles in flight with
// cp.async.bulk (the TMA engine, SASS UBLKCP): the tile's values, column indices and row pointers
// land in a shared-memory stage and signal an mbarrier with their byte count.  The other threads
// only gather x, multiply in place and reduce rows, so HBM streaming never waits for the gather /
// reduce phases of the same block.
constexpr int kPipeCap = 1792;  // entries per stage = 7 * kTileRows
#ifndef NXFX_SPMV_STAGES
#define NXFX_SPMV_STAGES 2
#endif
constexpr int kStages = NXFX_SPMV_STAGES;

struct alignas(128) SpmvStage {
  double vals[kPipeCap];
  int cols[kPipeCap];
  int rows[kTileRows + 8];
};

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
// streaming variant: the matrix is read once per product, so its lines are marked evict-first in
// L2 and do not push out the x vector the gathers keep re-using
__device__ __forceinline__ uint64_t l2_evict_first_policy() {
  uint64_t p;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
  return p;
}
__device__ __forceinline__ void bulk_g2s_stream(void* dst, const void* src, uint32_t bytes, uint64_t* bar,
                                                uint64_t policy) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(
          smem_u32(dst)),
      "l"(src), "r"(bytes), "r"(smem_u32(bar)), "l"(policy)
      : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok = 0;
  const uint32_t addr = smem_u32(bar);
  while (!ok) {
    asm volatile(
        "{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}"
        : "=r"(ok)
        : "r"(addr), "r"(parity)
        : "memory");
  }
}

// tile_base[t] = rowptr[t * kTileRows], tile_base[ntiles] = nnz
__global__ void __launch_bounds__(kThreads)
tile_base_kernel(int n, int ntiles, const int32_t* __restrict__ rowptr, int32_t* __restrict__ tile_base,
                 int32_t* __restrict__ max_tile_nnz) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t > ntiles) return;
  const int r = min(t * kTileRows, n);
  const int b = rowptr[r];
  tile_base[t] = b;
  if (t < ntiles) atomicMax(max_tile_nnz, rowptr[min(r + kTileRows, n)] - b);
}

template <int MODE>
__global__ void __launch_bounds__(kTileRows)
spmv_pipe_kernel(int n, int ntiles, const int32_t* __restrict__ rowptr,
                 const int32_t* __restrict__ colidx, const double* __restrict__ vals,
                 const int32_t* __restrict__ tile_base, const double* __restrict__ x,
                 double* __restrict__ y, const double* __restrict__ b, double* partial,
                 unsigned int* ticket, double* norm2_out, int loff = 0,
                 const double* __restrict__ w_r = nullptr, const double* __restrict__ w_b = nullptr,
                 PeerDev pc = PeerDev{}, const int32_t* __restrict__ shared_lm = nullptr, int n_shared = 0,
                 double* lam_scratch = nullptr) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  SpmvStage* st = reinterpret_cast<SpmvStage*>(smem_raw);
  uint64_t* full = reinterpret_cast<uint64_t*>(smem_raw + kStages * sizeof(SpmvStage));
  __shared__ double red[kTileRows / 32];
  const int tid = threadIdx.x;
  if (tid == 0) {
    for (int s = 0; s < kStages; ++s) mbar_init(full + s, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }
  __syncthreads();
  const uint64_t stream_policy = l2_evict_first_policy();
  auto issue = [&](int tile, int s) {
    const int r0 = tile * kTileRows;
    const int nr = min(kTileRows, n - r0);
    const int sb = tile_base[tile], se = tile_base[tile + 1];
    const int s4 = sb & ~3;
    const int cnt4 = ((se + 3) & ~3) - s4;
    const uint32_t rbytes = (uint32_t)(((nr + 1) * 4 + 15) & ~15);
    mbar_expect_tx(full + s, (uint32_t)cnt4 * 12u + rbytes);
    if (cnt4 > 0) {
      bulk_g2s_stream(st[s].vals, vals + s4, (uint32_t)cnt4 * 8u, full + s, stream_policy);
      bulk_g2s_stream(st[s].cols, colidx + s4, (uint32_t)cnt4 * 4u, full + s, stream_policy);
    }
    bulk_g2s_stream(st[s].rows, rowptr + r0, rbytes, full + s, stream_policy);
  };
  if (tid == 0) {
    for (int k = 0; k < kStages - 1; ++k) {
      const int tile = blockIdx.x + k * gridDim.x;
      if (tile < ntiles) issue(tile, k);
    }
  }
  // Programmatic dependent launch: everything above only touches the matrix (complete long before
  // the preceding kernel started); x, b, y and the reduction scratch are used below.  A no-op when
  // the kernel was launched without the attribute.
  asm volatile("griddepcontrol.wait;" ::: "memory");
  double nrm = 0.0, nrb = 0.0;
  int it = 0;
  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++it) {
    const int s = it % kStages;
    if (tid == 0) {
      const int pre = tile + (kStages - 1) * gridDim.x;
      if (pre < ntiles) {
        // the stage being refilled was multiplied in place by generic-proxy stores
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        issue(pre, (it + kStages - 1) % kStages);
      }
    }
    const int r0 = tile * kTileRows;
    const int nr = min(kTileRows, n - r0);
    double bi = 0.0;
    if (MODE >= 1 && tid < nr) bi = __ldcs(b + r0 + tid);
    mbar_wait(full + s, (uint32_t)((it / kStages) & 1));
    SpmvStage& S = st[s];
    const int base = S.rows[0];
    const int off = base & 3;
    const int tnnz = S.rows[nr] - base;
    constexpr int kPer = kPipeCap / kTileRows;
    int c[kPer];
    double xv[kPer];
#pragma unroll
    for (int k = 0; k < kPer; ++k) {
      const int idx = tid + k * kTileRows;
      if (idx < tnnz) c[k] = S.cols[off + idx];
    }
#pragma unroll
    for (int k = 0; k < kPer; ++k) {
      const int idx = tid + k * kTileRows;
      if (idx < tnnz) xv[k] = x[c[k]];
    }
#pragma unroll
    for (int k = 0; k < kPer; ++k) {
      const int idx = tid + k * kTileRows;
      if (idx < tnnz) S.vals[off + idx] = __dmul_rn(S.vals[off + idx], xv[k]);
    }
    __syncthreads();
    if (tid < nr) {
      const int rs = S.rows[tid] - base + off, re = S.rows[tid + 1] - base + off;
      double acc = 0.0;
      for (int k = rs; k < re; ++k) acc = __dadd_rn(acc, S.vals[k]);
      if (MODE == 0) {
        y[r0 + tid] = acc;
      } else {
        const double r = __dsub_rn(bi, acc);
        if (y) y[r0 + tid] = r;  // y == nullptr: norms only
        if (MODE >= 2 && r0 + tid >= loff) {  // multi-GPU: weighted multiplier rows
          const double wr = w_r[r0 + tid - loff];
          nrm += wr * r * r;
          nrb += w_b[r0 + tid - loff] * bi * bi;
          // replicated rows (weight 0 on every rank) hold partial sums: parked for the exchange below
          if (MODE == 3 && wr == 0.0) lam_scratch[r0 + tid - loff] = r;
        } else {
          nrm += r * r;
          nrb += bi * bi;
        }
      }
    }
    // order this thread's generic-proxy accesses to the stage before the TMA refill
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    __syncthreads();
  }
  if (MODE >= 1 && MODE < 3) {
    double mine[2] = {block_sum<kTileRows>(nrm, red), block_sum<kTileRows>(nrb, red)};
    finish_partials<kTileRows, 2>(mine, partial, gridDim.x, ticket, norm2_out, red);
  }
  if (MODE == 3) {
    __shared__ double loc[2];
    double mine[2] = {block_sum<kTileRows>(nrm, red), block_sum<kTileRows>(nrb, red)};
    if (!finish_partials<kTileRows, 2>(mine, partial, gridDim.x, ticket, loc, red)) return;
    __syncthreads();  // loc[] written by thread 0
    peer_ll_send(pc, 1, n_shared + 2,
                 [&](int i) { return i < n_shared ? __ldcg(lam_scratch + shared_lm[i]) : loc[i - n_shared]; });
    double acc = 0.0;
    for (int i = tid; i < n_shared; i += kTileRows) {
      double v = 0.0;
      for (int src = 0; src < pc.nranks; ++src) v += peer_ll_recv(pc, 1, src, i);  // rank order
      if (y) y[loff + shared_lm[i]] = v;
      acc += v * v;
    }
    acc = block_sum<kTileRows>(acc, red);
    if (tid == 0) {
      double s0 = acc, s1 = 0.0;
      for (int src = 0; src < pc.nranks; ++src) {
        s0 += peer_ll_recv(pc, 1, src, n_shared);
        s1 += peer_ll_recv(pc, 1, src, n_shared + 1);
      }
      norm2_out[0] = s0;
      norm2_out[1] = s1;
    }
  }
}

// ---- vector kernels --------------------------------------------------------------------------
// out[k] = <a_k, w>, k < K, a_k = A + k*stride (one pass over w)
template <int K>
__global__ void __launch_bounds__(kThreads)
multi_dot_kernel(int n, const double* __restrict__ A, size_t stride, const double* __restrict__ w,
                 double* partial, unsigned int* ticket, double* out) {
  __shared__ double red[kThreads / 32];
  double acc[K];
#pragma unroll
  for (int k = 0; k < K; ++k) acc[k] = 0.0;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const double wi = w[i];
#pragma unroll
    for (int k = 0; k < K; ++k) acc[k] += A[(size_t)k * stride + i] * wi;
  }
  double mine[K];
#pragma unroll
  for (int k = 0; k < K; ++k) mine[k] = block_sum<kThreads>(acc[k], red);
  finish_partials<kThreads, K>(mine, partial, gridDim.x, ticket, out, red);
}

// out[0] = sum w1_i r_i^2, out[1] = sum w2_i b_i^2 in one pass (weights 1 for i < loff, w[i - loff] on the
// multiplier rows; multi-GPU residual:
// w1 excludes every replicated multiplier row -- their partial sums are O(1) and only cancel in the
// all-reduce, so they must never enter a local norm -- w2 counts owned rows).  pw (nullptr: none): extra weight of the rows p0 .. p0 + np - 1 in both sums -- 0 on
// the nodal pressure rows of the shared bifurcations (continuous pressure), partial sums like the multiplier rows
__global__ void __launch_bounds__(kThreads)
weighted_norm2_pair_kernel(int n, int loff, const double* __restrict__ r, const double* __restrict__ w1,
                           const double* __restrict__ b, const double* __restrict__ w2, double* partial,
                           unsigned int* ticket, double* out, int p0 = 0, int np = 0,
                           const double* __restrict__ pw = nullptr) {
  __shared__ double red[kThreads / 32];
  double a1 = 0.0, a2 = 0.0;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const double ri = r[i], bi = b[i];
    const bool lam = i >= loff;
    const double wp = (pw && i >= p0 && i < p0 + np) ? pw[i - p0] : 1.0;
    a1 += (lam ? w1[i - loff] : wp) * ri * ri;
    a2 += (lam ? w2[i - loff] : wp) * bi * bi;
  }
  double mine[2] = {block_sum<kThreads>(a1, red), block_sum<kThreads>(a2, red)};
  finish_partials<kThreads, 2>(mine, partial, gridDim.x, ticket, out, red);
}

// w += sum_k sign * h[k] * a_k
template <int K>
__global__ void __launch_bounds__(kThreads)
multi_axpy_kernel(int n, const double* __restrict__ A, size_t stride, const double* __restrict__ h,
                  double sign, double* __restrict__ w) {
  double hk[K];
#pragma unroll
  for (int k = 0; k < K; ++k) hk[k] = sign * h[k];
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    double wi = w[i];
#pragma unroll
    for (int k = 0; k < K; ++k) wi += hk[k] * A[(size_t)k * stride + i];
    w[i] = wi;
  }
}

// y = x * (1 / sqrt(*norm2))   (normalise a Krylov vector with a device-side norm)
__global__ void __launch_bounds__(kThreads)
scale_by_inv_norm_kernel(int n, const double* __restrict__ x, const double* norm2,
                         double* __restrict__ y) {
  const double s = 1.0 / sqrt(*norm2);
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
    y[i] = x[i] * s;
}

// out = (or +=) in with the entries from `off` on multiplied by s (constraint rows of a k-fold accumulated matrix)
template <bool ADD>
__global__ void __launch_bounds__(kThreads)
scale_tail_kernel(int n, int off, double s, const double* __restrict__ in, double* __restrict__ out) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const double v = i < off ? in[i] : in[i] * s;
    if (ADD) out[i] += v; else out[i] = v;
  }
}

__global__ void __launch_bounds__(kThreads)
add_kernel(int n, const double* __restrict__ z, double* __restrict__ x) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
    x[i] += z[i];
}

}  // namespace nxfx
