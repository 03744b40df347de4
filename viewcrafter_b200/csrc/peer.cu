// Multi-GPU exchange kernels over NVLink peer memory (one process per GPU; the buffers of the other ranks are mapped into
// this process through CUDA IPC by the Python side, viewcrafter_b200/parallel.py).  New functionality -- the reference is
// single-GPU (SURVEY.md 8e): the frame-sharded U-Net switches between the "frame" layout [(b, t_local, hw), C] of the spatial
// ops and the "site" layout [(b, t_all, hw_local), C] of the temporal ops 78 times per forward.
//
//   peer_exchange_kernel   ONE kernel per layout switch: every rank reads its local activation once and stores each row
//                          straight into the receive buffer of the rank that owns it in the other layout (16-byte stores
//                          through the NVLink aperture); while the rows stream through the registers it also accumulates the
//                          GroupNorm(32) statistics of the tensor (the op that follows every frames->sites switch is a 5-D
//                          GroupNorm whose statistics span all ranks) and publishes its partial sums to every peer.  No pack
//                          / unpack copies, no NCCL call, no separate statistics pass, no all-reduce.
//   gn_peer_allreduce_kernel  the same publish / wait step alone, for the GroupNorms in the middle of a temporal block.
//
// Synchronisation: every collective has a sequence number (a device-side counter, so that a captured CUDA graph can be
// replayed).  The last CTA of rank r to finish stores the number into slot r of every peer's flag array with release.sys
// semantics after a system-scope fence, then waits (acquire.sys) until its own flag array shows the number for every peer:
// when the kernel ends, the data of all peers has landed.  Receive buffers are reused: a rank can only be writing collective
// s into a peer's buffer after that peer signalled s-1, which in the peer's stream order comes after every reader of the
// previous contents (the two directions use different buffers and strictly alternate).
#include <cstring>

#include "common.cuh"
#include "kernels.h"

namespace vc {

static constexpr int PEER_MAX = 8;
static constexpr int PEER_BMAX = 4;                 // batch samples per rank (vc_peer_comm.Bmax): e.g. the three branches of three-way CFG
static constexpr int PEER_ALLREDUCE_THREADS = 128;  // gn_peer_allreduce_kernel block (peer_finish loops over the B*64 sums)
static_assert(PEER_ALLREDUCE_THREADS >= PEER_MAX, "peer_finish: one thread per rank signals / waits");

struct PeerCommDev {
  int world, rank;
  unsigned int* flags;                 // own [world]
  unsigned int* peer_flags[PEER_MAX];  // rank p's flag array as mapped here (p == rank: own)
  unsigned int* seq;                   // own: number of collectives completed
  unsigned int* done;                  // own: CTA completion counter of the running collective
  float* stats_slots[PEER_MAX];        // rank p's [2][Bmax][world][64] partial-statistics slots
  float* cur_stats;                    // own [Bmax][world][64]: the gathered statistics of the last collective
  int Bmax;
};

struct ExchangeParams {
  const __half* src;
  __half* dst[PEER_MAX];
  int B, T, HW, HWl, C, vecs, ppi, cg;
  int f0[PEER_MAX + 1];
  int to_sites, with_stats;
  long long rows_local;                // rows per batch sample in the source layout
  int splits;
  long long rows_per_split;
  float* partial;                      // [B][splits][64]
  PeerCommDev pc;
};

__device__ __forceinline__ void st_release_sys(unsigned int* p, unsigned int v) {
  asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ unsigned int ld_acquire_sys(const unsigned int* p) {
  unsigned int v;
  asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}

// Tail of every collective, executed by ALL threads of the LAST CTA of this rank (the caller has established that every other
// CTA's stores are fenced): publish this rank's B*64 partial sums (the sum over `splits` of partial[b][split][64]; nothing when
// !with_stats), signal, wait for all peers, gather their sums.  Strided over B*64 values, so any block size covers up to PEER_BMAX
// samples; the signal / wait step needs blockDim.x >= world (checked on the host before every launch).
__device__ __forceinline__ void peer_finish(const PeerCommDev& pc, int B, bool with_stats, const float* partial, int splits, int tid) {
  const unsigned int s = *reinterpret_cast<volatile unsigned int*>(pc.seq) + 1u;
  const int n = B * 64;
  const int parity = (int)(s & 1u);
  if (with_stats) {
    for (int i = tid; i < n; i += blockDim.x) {
      const int b = i >> 6, t = i & 63;
      float mine = 0.f;
      for (int sp = 0; sp < splits; ++sp) mine += __ldcg(partial + ((long long)b * splits + sp) * 64 + t);
      const long long slot = (((long long)parity * pc.Bmax + b) * pc.world + pc.rank) * 64 + t;
      for (int q = 0; q < pc.world; ++q) pc.stats_slots[q][slot] = mine;
    }
  }
  __threadfence_system();
  __syncthreads();
  if (tid < pc.world) {
    st_release_sys(pc.peer_flags[tid] + pc.rank, s);
    // bounded wait (~30 s): a rank that never arrives (crashed peer, mismatched call sequence) must not hang the GPU
    unsigned long long spins = 0;
    while ((int)(ld_acquire_sys(pc.flags + tid) - s) < 0) {
      __nanosleep(spins < 1024 ? 32 : 256);
      if (++spins > 120000000ull) __trap();
    }
  }
  __syncthreads();
  if (with_stats) {
    __threadfence_system();
    const float* own = pc.stats_slots[pc.rank] + (long long)parity * pc.Bmax * pc.world * 64;
    for (int i = tid; i < B * pc.world * 64; i += blockDim.x) pc.cur_stats[i] = __ldcg(own + i);
  }
  if (tid == 0) {
    *pc.done = 0u;
    *pc.seq = s;
  }
}

__device__ __forceinline__ void acc8(const uint4& u, float (&s)[8], float (&ss)[8]) {
  const __half2* h = reinterpret_cast<const __half2*>(&u);
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    const float2 f = __half22float2(h[e]);
    s[2 * e] += f.x; ss[2 * e] = fmaf(f.x, f.x, ss[2 * e]);
    s[2 * e + 1] += f.y; ss[2 * e + 1] = fmaf(f.y, f.y, ss[2 * e + 1]);
  }
}

__global__ void __launch_bounds__(512) peer_exchange_kernel(const __grid_constant__ ExchangeParams p) {
  extern __shared__ float red[];   // [ppi][2*C] (with_stats): fixed-order reduction, no float atomics
  __shared__ int is_last;
  const int tid = threadIdx.x;
  const int v = tid % p.vecs, pl = tid / p.vecs;
  const int split = blockIdx.x, b = blockIdx.y;
  float s[8], ss[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) s[e] = ss[e] = 0.f;
  const long long r0 = (long long)split * p.rows_per_split;
  const long long r1 = min(p.rows_local, r0 + p.rows_per_split);
  const __half* sp = p.src + ((long long)b * p.rows_local) * p.C + v * 8;
  const int me = p.pc.rank;
  // destination of a source row
  auto route = [&](long long r, int& peer) -> long long {
    if (p.to_sites) {                                  // r = tl * HW + hw
      const int tl = (int)(r / p.HW);
      const int hw = (int)(r - (long long)tl * p.HW);
      peer = hw / p.HWl;
      return ((long long)b * p.T + p.f0[me] + tl) * p.HWl + (hw - peer * p.HWl);
    }
    const int t = (int)(r / p.HWl);                    // r = t * HWl + s
    const int sidx = (int)(r - (long long)t * p.HWl);
    int q = 0;
    while (t >= p.f0[q + 1]) ++q;
    peer = q;
    const int tlq = p.f0[q + 1] - p.f0[q];
    return ((long long)b * tlq + (t - p.f0[q])) * p.HW + (long long)me * p.HWl + sidx;
  };
  long long r = r0 + pl;
  for (; r + 3ll * p.ppi < r1; r += 4ll * p.ppi) {     // 4 independent 16-byte loads in flight per thread
    uint4 u[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) u[i] = *reinterpret_cast<const uint4*>(sp + (r + (long long)i * p.ppi) * p.C);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      int peer;
      const long long drow = route(r + (long long)i * p.ppi, peer);
      *reinterpret_cast<uint4*>(p.dst[peer] + drow * p.C + v * 8) = u[i];
      if (p.with_stats) acc8(u[i], s, ss);
    }
  }
  for (; r < r1; r += p.ppi) {
    const uint4 u = *reinterpret_cast<const uint4*>(sp + r * p.C);
    int peer;
    const long long drow = route(r, peer);
    *reinterpret_cast<uint4*>(p.dst[peer] + drow * p.C + v * 8) = u;
    if (p.with_stats) acc8(u, s, ss);
  }
  if (p.with_stats) {
    float* mine = red + (long long)pl * 2 * p.C;
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      mine[v * 8 + e] = s[e];
      mine[p.C + v * 8 + e] = ss[e];
    }
    __syncthreads();
    if (tid < 64) {
      const int grp = tid >> 1, which = tid & 1;
      float acc = 0.f;
      for (int q = 0; q < p.ppi; ++q) {
        const float* row = red + (long long)q * 2 * p.C + which * p.C;
        for (int c = grp * p.cg; c < (grp + 1) * p.cg; ++c) acc += row[c];
      }
      p.partial[((long long)b * p.splits + split) * 64 + tid] = acc;
    }
  }
  // ---- completion: the last CTA of this rank runs the signal / wait protocol ----
  __threadfence_system();
  __syncthreads();
  if (tid == 0) {
    const unsigned int d = atomicAdd(p.pc.done, 1u);
    is_last = (d == gridDim.x * gridDim.y - 1u) ? 1 : 0;
    __threadfence();
  }
  __syncthreads();
  if (!is_last) return;
  peer_finish(p.pc, p.B, p.with_stats != 0, p.partial, p.splits, tid);
}

// (sum, sumsq) per group of this rank's rows -> every rank's slots -> cur_stats[B][world][64]
// B == 0: the signal / wait step alone -- the completion barrier of a layout switch that a GEMM's epilogue performed (its TMA stores to
// the peers are complete when that kernel ends; this kernel, next in the stream, fences and publishes the sequence number).
__global__ void __launch_bounds__(PEER_ALLREDUCE_THREADS) gn_peer_allreduce_kernel(const float* __restrict__ partial, int splits, int B,
                                                                                const __grid_constant__ PeerCommDev pc) {
  peer_finish(pc, B, B > 0, partial, splits, threadIdx.x);
}

}  // namespace vc

// ------------------------------------------------------------------------------------------------------------------
#include "../../include/vc_b200.h"

namespace vc {
int groupnorm_stats_partials(const __half* x1, int C1, int samples, long long rows_per_sample, float* partial_ws, size_t ws_bytes,
                             int* splits_out, cudaStream_t stream);

static int to_dev(const vc_peer_comm* c, PeerCommDev& d) {
  VC_REQUIRE(c && c->world >= 1 && c->world <= PEER_MAX && c->rank >= 0 && c->rank < c->world, "peer comm: bad world / rank");
  VC_REQUIRE(c->flags && c->seq && c->done && c->cur_stats && c->Bmax >= 1 && c->Bmax <= PEER_BMAX,
             "peer comm: null buffer or Bmax not in 1..%d", PEER_BMAX);
  d.world = c->world; d.rank = c->rank;
  d.flags = reinterpret_cast<unsigned int*>(c->flags);
  d.seq = reinterpret_cast<unsigned int*>(c->seq);
  d.done = reinterpret_cast<unsigned int*>(c->done);
  d.cur_stats = reinterpret_cast<float*>(c->cur_stats);
  d.Bmax = c->Bmax;
  for (int q = 0; q < c->world; ++q) {
    VC_REQUIRE(c->peer_flags[q] && c->stats_slots[q], "peer comm: unmapped peer %d", q);
    d.peer_flags[q] = reinterpret_cast<unsigned int*>(c->peer_flags[q]);
    d.stats_slots[q] = reinterpret_cast<float*>(c->stats_slots[q]);
  }
  return VC_OK;
}
}  // namespace vc

extern "C" {

int vc_enable_peer_access(int32_t peer_device) {
  int dev = 0;
  VC_CHECK_CUDA(cudaGetDevice(&dev));
  if (dev == peer_device) return VC_OK;
  int can = 0;
  VC_CHECK_CUDA(cudaDeviceCanAccessPeer(&can, dev, peer_device));
  if (!can) { vc::set_error("device %d cannot access peer %d", dev, peer_device); return VC_ERR_UNSUPPORTED; }
  cudaError_t e = cudaDeviceEnablePeerAccess(peer_device, 0);
  if (e == cudaErrorPeerAccessAlreadyEnabled) { (void)cudaGetLastError(); return VC_OK; }
  VC_CHECK_CUDA(e);
  return VC_OK;
}

/* IPC-shareable device memory: plain cudaMalloc (the handle then refers to exactly this allocation), zero-filled.  The importing
 * rank opens the handle with ITS OWN compute device current, so that the lazy peer mapping is created for the device whose
 * kernels will dereference the pointer. */
int vc_peer_alloc(size_t bytes, void** ptr, void* handle64) {
  if (!ptr || !handle64 || bytes == 0) { vc::set_error("vc_peer_alloc: bad args"); return VC_ERR_ARG; }
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "cudaIpcMemHandle_t is 64 bytes");
  void* p = nullptr;
  VC_CHECK_CUDA(cudaMalloc(&p, bytes));
  VC_CHECK_CUDA(cudaMemset(p, 0, bytes));
  VC_CHECK_CUDA(cudaDeviceSynchronize());
  cudaIpcMemHandle_t h;
  cudaError_t e = cudaIpcGetMemHandle(&h, p);
  if (e != cudaSuccess) {
    cudaFree(p);
    vc::set_error("cudaIpcGetMemHandle failed: %s", cudaGetErrorString(e));
    return VC_ERR_CUDA;
  }
  memcpy(handle64, &h, 64);
  *ptr = p;
  return VC_OK;
}
int vc_peer_open(const void* handle64, void** ptr) {
  if (!ptr || !handle64) { vc::set_error("vc_peer_open: bad args"); return VC_ERR_ARG; }
  cudaIpcMemHandle_t h;
  memcpy(&h, handle64, 64);
  VC_CHECK_CUDA(cudaIpcOpenMemHandle(ptr, h, cudaIpcMemLazyEnablePeerAccess));
  return VC_OK;
}
int vc_peer_close(void* ptr) {
  VC_CHECK_CUDA(cudaIpcCloseMemHandle(ptr));
  return VC_OK;
}
int vc_peer_free(void* ptr) {
  VC_CHECK_CUDA(cudaFree(ptr));
  return VC_OK;
}

int vc_peer_exchange(const vc_peer_comm* c, const void* src, void* const* dst, int32_t to_sites, int32_t B, int32_t T, int32_t HW,
                     int32_t C, const int32_t* f0, int32_t with_stats, void* ws, size_t ws_bytes, void* stream) {
  using namespace vc;
  ExchangeParams p;
  memset(&p, 0, sizeof(p));
  int rc = to_dev(c, p.pc);
  if (rc) return rc;
  VC_REQUIRE(src && dst && f0 && B >= 1 && B <= c->Bmax && T >= 1 && HW >= 1 && HW % c->world == 0, "peer_exchange: bad shape");
  VC_REQUIRE(C % 32 == 0 && C <= 4096, "peer_exchange: unsupported C=%d", C);
  VC_REQUIRE(f0[0] == 0 && f0[c->world] == T, "peer_exchange: frame ranges must cover [0, T)");
  p.src = reinterpret_cast<const __half*>(src);
  for (int q = 0; q < c->world; ++q) { VC_REQUIRE(dst[q], "peer_exchange: null destination"); p.dst[q] = reinterpret_cast<__half*>(dst[q]); }
  for (int q = 0; q <= c->world; ++q) p.f0[q] = f0[q];
  p.B = B; p.T = T; p.HW = HW; p.HWl = HW / c->world; p.C = C;
  p.vecs = C / 8; p.ppi = 512 / p.vecs > 0 ? 512 / p.vecs : 1; p.cg = C / 32;
  p.to_sites = to_sites; p.with_stats = with_stats && to_sites;
  const int tl = f0[c->rank + 1] - f0[c->rank];
  p.rows_local = to_sites ? (long long)tl * HW : (long long)T * p.HWl;
  VC_REQUIRE(p.rows_local > 0, "peer_exchange: this rank owns no rows");
  int splits = (2 * sm_count() + B - 1) / B;
  const long long max_useful = (p.rows_local + p.ppi - 1) / p.ppi;
  if (splits > max_useful) splits = (int)max_useful;
  if (splits > 512) splits = 512;
  if (splits < 1) splits = 1;
  p.splits = splits;
  p.rows_per_split = (p.rows_local + splits - 1) / splits;
  p.partial = reinterpret_cast<float*>(ws);
  VC_REQUIRE(!p.with_stats || (ws && ws_bytes >= (size_t)B * splits * 64 * sizeof(float)), "peer_exchange: workspace too small");
  // the last CTA runs peer_finish: its threads loop over the B*64 sums, and one thread per rank signals / waits
  VC_REQUIRE(p.vecs * p.ppi >= c->world && B <= PEER_BMAX, "peer_exchange: block of %d threads for world %d, B %d", p.vecs * p.ppi, c->world, B);
  dim3 grid(splits, B);
  peer_exchange_kernel<<<grid, p.vecs * p.ppi, p.with_stats ? (size_t)2 * C * p.ppi * sizeof(float) : 0, reinterpret_cast<cudaStream_t>(stream)>>>(p);
  VC_CHECK_CUDA(cudaGetLastError());
  return VC_OK;
}

int vc_peer_groupnorm_stats(const vc_peer_comm* c, const void* x, int32_t C, int32_t samples, int64_t rows_per_sample, void* ws,
                            size_t ws_bytes, void* stream) {
  using namespace vc;
  PeerCommDev d;
  int rc = to_dev(c, d);
  if (rc) return rc;
  VC_REQUIRE(samples >= 1 && samples <= c->Bmax, "peer_groupnorm_stats: samples %d exceed Bmax %d", samples, c->Bmax);
  int splits = 0;
  rc = groupnorm_stats_partials(reinterpret_cast<const __half*>(x), C, samples, rows_per_sample, reinterpret_cast<float*>(ws), ws_bytes,
                                &splits, reinterpret_cast<cudaStream_t>(stream));
  if (rc) return rc;
  gn_peer_allreduce_kernel<<<1, PEER_ALLREDUCE_THREADS, 0, reinterpret_cast<cudaStream_t>(stream)>>>(reinterpret_cast<const float*>(ws), splits, samples, d);
  VC_CHECK_CUDA(cudaGetLastError());
  return VC_OK;
}

/* completion of a layout switch performed by a GEMM epilogue (vc_gemm_desc.peer): the per-group sums of the tensor just written -- from the
 * GEMM's gn_part records, summed over this rank's rows -- are published to every rank and the ranks rendezvous; afterwards every peer's
 * tiles have landed in this rank's receive buffer and cur_stats holds the [samples][world][32][2] sums for vc_groupnorm_apply_parts.
 * geom == NULL: rendezvous only (sites -> frames: no cross-rank statistics follow). */
int vc_peer_finish_scatter(const vc_peer_comm* c, const vc_gn_part_geom* geom, int32_t C, int32_t samples, void* ws, size_t ws_bytes, void* stream) {
  using namespace vc;
  PeerCommDev d;
  int rc = to_dev(c, d);
  if (rc) return rc;
  int splits = 0, B = 0;
  if (geom) {
    VC_REQUIRE(samples >= 1 && samples <= c->Bmax, "peer_finish_scatter: samples %d exceed Bmax %d", samples, c->Bmax);
    GnPartGeom g;
    g.part = geom->part; g.n_chunks = geom->n_chunks; g.sub = geom->sub; g.rb_per_z = geom->rb_per_z; g.samples_per_z = geom->samples_per_z;
    g.rb_per_sample = geom->rb_per_sample;
    rc = groupnorm_parts_to_partials(g, C, samples, reinterpret_cast<float*>(ws), ws_bytes, &splits, reinterpret_cast<cudaStream_t>(stream));
    if (rc) return rc;
    B = samples;
  }
  gn_peer_allreduce_kernel<<<1, PEER_ALLREDUCE_THREADS, 0, reinterpret_cast<cudaStream_t>(stream)>>>(reinterpret_cast<const float*>(ws), splits, B, d);
  VC_CHECK_CUDA(cudaGetLastError());
  return VC_OK;
}

}  // extern "C"
