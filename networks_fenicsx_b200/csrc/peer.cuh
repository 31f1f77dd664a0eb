// Peer exchange over NVLink for the partitioned (multi-GPU) solve.
//
// What couples the ranks of a partitioned network is additive and tiny: the partial pivots / link
// conductances / right-hand sides of the SHARED nodes of the elimination tree (3 x (world - 1) doubles for
// a balanced binary tree) and the shared multiplier rows of a residual with two norm partials.  Instead
// of returning to the host for an NCCL all-reduce, the kernel that produces the partial sums stores them
// straight into EVERY rank's exchange buffer (cudaIpc-mapped peer memory; the stores travel over NVLink /
// NVSwitch), polls its own buffer for the contributions of all ranks and adds them up in rank order --
// the same order on every rank, so all ranks continue with bit-identical values (identical shared nodes,
// identical norms, identical refinement decisions) and the whole solve keeps the single-GPU launch
// sequence with no host round trip.
//
// Buffer of one rank (cudaMalloc, exported with cudaIpcGetMemHandle):
//   [0, 256)   reserved
//   [256, ..)  u64 words[kPeerChannels][2][nranks][slot]   parity = epoch & 1, slot = 2 words per value
// Two parities suffice: a rank can only deliver epoch e+2 after it has consumed everybody's e+1,
// which everybody sends only after consuming epoch e.
#pragma once

#include <cstdint>

namespace nxfx {

constexpr int kMaxPeers = 16;
constexpr int kPeerChannels = 2;  // 0: top chunk of the tree solve, 1: residual
constexpr size_t kPeerHeaderBytes = 256;

struct PeerDev {
  unsigned long long base[kMaxPeers];  // exchange buffer of every rank as seen from this device
  int rank, nranks;                    // nranks <= 1: single GPU, no exchange
  int slot;                            // 8-byte words per (channel, parity, source)
  unsigned int epoch;                  // of this use of the channel (starts at 1)
  int* err;                            // mapped host word: set to 1 when a peer did not arrive in time
};

__device__ __forceinline__ double* peer_data(const PeerDev& c, int dst, int ch, int src) {
  char* b = reinterpret_cast<char*>(c.base[dst]) + kPeerHeaderBytes;
  return reinterpret_cast<double*>(b) + ((size_t)((ch * 2 + (int)(c.epoch & 1u)) * c.nranks + src)) * (size_t)c.slot;
}

// Low-latency form (what NCCL calls the LL protocol): every double travels as two 8-byte words
// {high 32 bits | epoch}, {low 32 bits | epoch}.  An aligned 8-byte store is single-copy atomic, so the
// epoch in a word says that ITS payload has arrived: no fence, no separate flag, no second round trip -- the
// receiver just polls the words it needs.  Cost: one NVLink store latency (measured: the fence + flag form
// took >= 6 us per exchange between two B200s, about twice this).
__device__ __forceinline__ unsigned long long* peer_words(const PeerDev& c, int dst, int ch, int src) {
  return reinterpret_cast<unsigned long long*>(peer_data(c, dst, ch, src));  // 2 words per double: slot holds slot/2 doubles
}

// send get(i), i < n, to every rank (all threads of the calling block take part; no barrier needed)
template <typename Get>
__device__ __forceinline__ void peer_ll_send(const PeerDev& c, int ch, int n, Get get) {
  const unsigned long long ep = c.epoch;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const unsigned long long v = (unsigned long long)__double_as_longlong(get(i));
    const unsigned long long w0 = (v & 0xFFFFFFFF00000000ull) | ep, w1 = (v << 32) | ep;
    for (int dst = 0; dst < c.nranks; ++dst) {
      unsigned long long* out = peer_words(c, dst, ch, c.rank) + 2 * i;
      asm volatile("st.volatile.global.u64 [%0], %1;" ::"l"(out), "l"(w0) : "memory");
      asm volatile("st.volatile.global.u64 [%0], %1;" ::"l"(out + 1), "l"(w1) : "memory");
    }
  }
}

// element i of rank src's contribution to this epoch (spins until both words carry the epoch)
__device__ __forceinline__ double peer_ll_recv(const PeerDev& c, int ch, int src, int i) {
  const unsigned long long ep = c.epoch;
  const unsigned long long* in = peer_words(c, c.rank, ch, src) + 2 * i;
  unsigned long long w0, w1, t0 = 0, t1;
  while (true) {
    asm volatile("ld.volatile.global.u64 %0, [%1];" : "=l"(w0) : "l"(in) : "memory");
    asm volatile("ld.volatile.global.u64 %0, [%1];" : "=l"(w1) : "l"(in + 1) : "memory");
    if ((w0 & 0xFFFFFFFFull) == ep && (w1 & 0xFFFFFFFFull) == ep) break;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
    if (t0 == 0) t0 = t1;
    if (t1 - t0 > 4000000000ull) {  // 4 s: a peer is gone -- flag the error and let the kernel finish
      *reinterpret_cast<volatile int*>(c.err) = 1;
      break;
    }
  }
  return __longlong_as_double((long long)((w0 & 0xFFFFFFFF00000000ull) | (w1 >> 32)));
}

// ---- in-process all-reduce (nxfx_group_sum) ----------------------------------------------------------
// Ranks that are threads of one process reduce the split phases' buffers by reading each other's device
// memory directly; the host orders producers and consumers with events.  Every rank adds the
// contributions in rank order, so all ranks hold bit-identical sums.
struct GroupSrc {
  const double* p[kMaxPeers];
};

constexpr int kGroupSumThreads = 256;

__global__ void __launch_bounds__(kGroupSumThreads)
group_sum_kernel(GroupSrc src, int nranks, double* __restrict__ dst, int64_t n) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    double s = src.p[0][i];
#pragma unroll
    for (int r = 1; r < kMaxPeers; ++r)  // static indices: the pointers stay in the parameter bank (no stack copy)
      if (r < nranks) s += src.p[r][i];
    dst[i] = s;
  }
}

}  // namespace nxfx
