// gar_engine.cu — CUDA backend (sm_100a) and C ABI of the reconcile-diff engine.
//
// Implements include/garecon.h.  Stage logic lives in gar_rows.h / gar_pipeline.h; this file supplies what
// is specific to the GPU: kernels for the data-parallel stages, the device-wide exclusive scan, the stable LSD
// radix sort that orders hash-index buckets, device/pinned memory management, stream + event timing.
//
// There is deliberately no CPU path in this library: every entry point needs a live sm_100 device.

#include <cuda_runtime.h>
#include <unistd.h>

#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <atomic>
#include <exception>
#include <functional>
#include <mutex>
#include <thread>
#include <string>
#include <vector>
#include <utility>

#include "gar_pipeline.h"
#include "gar_shard.h"

#define GAR_VERSION_STRING "garecon 0.1.0 (sm_100a)"

// ------------------------------------------------------------------ kernels

template <class F>
__global__ void __launch_bounds__(256) k_for_each(const __grid_constant__ F f, u32 n) {
  u32 i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) f(i);
}

// Warp-synchronous variant: every lane of every warp calls f (padding lanes with valid = false), so f may vote.
template <class F, int MINB>
__global__ void __launch_bounds__(256, MINB) k_for_each_warp(const __grid_constant__ F f, u32 n) {
  u32 i = blockIdx.x * blockDim.x + threadIdx.x;
  f(i, i < n);
}
// tokenise_hostnames, staged (gar_pipeline.h FTokenise): with column-major slabs the hostnames of a block's 256 consecutive rows
// are ONE contiguous byte range.  One bulk copy (cp.async.bulk, completion on an mbarrier) brings it into shared memory and the
// rows are tokenised from there; a string outside the staged window (other layouts, a wider window) is read from the slab.
__device__ __forceinline__ u32 smem_addr(const void *p) { return (u32)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(u64 *bar, u32 count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_addr(bar)), "r"(count));
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(u64 *bar, u32 bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_addr(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tma_bulk_g2s(void *dst, const void *src, u32 bytes, u64 *bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_addr(dst)), "l"(src), "r"(bytes),
               "r"(smem_addr(bar))
               : "memory");
}
__device__ __forceinline__ void mbar_wait(u64 *bar, u32 parity) {
  u32 done;
  do {
    asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }" : "=r"(done) : "r"(smem_addr(bar)), "r"(parity) : "memory");
  } while (!done);
}
constexpr u32 TOK_STAGE_BYTES = 24 * 1024;  // 256 lbIngress hostnames of ~70 bytes
__global__ void __launch_bounds__(256) k_tokenise_staged(const __grid_constant__ FTokenise f, u32 n) {
  __shared__ alignas(128) u8 buf[TOK_STAGE_BYTES];
  __shared__ alignas(8) u64 bar;
  __shared__ u64 s_lo;
  __shared__ u32 s_bytes;
  const u32 r0 = blockIdx.x * blockDim.x, r1 = min(r0 + blockDim.x, n);
  const u8 *slab = f.T.o.slab;
  if (threadIdx.x == 0) {
    mbar_init(&bar, 1);
    const gar_str a = f.T.o.lbi_hostname[r0], b = f.T.o.lbi_hostname[r1 - 1];
    u64 lo = GAR_STR_OFF(a);
    const u64 hi = GAR_STR_OFF(b) + GAR_STR_LEN(b);
    u32 bytes = 0;
    if (hi > lo && (((uintptr_t)slab) & 15) == 0) {
      lo &= ~(u64)15;
      const u64 span = ((hi - lo + 15) & ~(u64)15) + 16;  // + slack for over-reads; slabs carry GAR_SLAB_PAD readable bytes behind their end
      bytes = (u32)(span < TOK_STAGE_BYTES ? span : TOK_STAGE_BYTES);
    }
    s_lo = lo;
    s_bytes = bytes;
    mbar_expect_tx(&bar, bytes);
    if (bytes) tma_bulk_g2s(buf, slab + lo, bytes, &bar);
  }
  __syncthreads();
  mbar_wait(&bar, 0);
  const u32 i = r0 + threadIdx.x;
  if (i >= n) return;
  const gar_str r = f.T.o.lbi_hostname[i];
  const u64 o = GAR_STR_OFF(r), len = GAR_STR_LEN(r);
  const bool staged = o >= s_lo && o + len + 16 <= s_lo + s_bytes;  // the 8-byte unaligned loads read up to 16 bytes past the end
  tokenise_hostname_at(f.T, f.W, i, Str{staged ? buf + (o - s_lo) : slab + o, (u32)len});
}

// Count on the device (an intermediate relation whose size the host never learns mid-diff): one element per thread over the
// buffer's CAPACITY; blocks beyond the real count leave at once.
template <class F>
__global__ void __launch_bounds__(256) k_for_each_dyn(const __grid_constant__ F f, const u32 *n_dev, u32 cap) {
  u32 n = *n_dev;
  if (n > cap) n = cap;
  u32 i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) f(i);
}
template <class F, int MINB>
__global__ void __launch_bounds__(256, MINB) k_for_each_warp_dyn(const __grid_constant__ F f, const u32 *n_dev, u32 cap) {
  u32 n = *n_dev;
  if (n > cap) n = cap;
  u32 i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < ((n + 31u) & ~31u)) f(i, i < n);  // whole warps enter or leave together
}
// Several row functors over their own tables in ONE launch (the index placement pass; the orphan count / emit passes):
// consecutive block ranges belong to consecutive functors.
template <class... Fs>
struct FPack;
template <>
struct FPack<> {
  __device__ __forceinline__ void call(int, u32) const {}
};
template <class F, class... R>
struct FPack<F, R...> {
  F f;
  FPack<R...> rest;
  FPack(const F &f_, const R &...r) : f(f_), rest(r...) {}
  __device__ __forceinline__ void call(int k, u32 i) const {
    if (k == 0) f(i);
    else rest.call(k - 1, i);
  }
};
constexpr int MULTI_MAX = 8;
struct MultiRanges {
  u32 blk_end[MULTI_MAX], n[MULTI_MAX];
  int count;
};
template <class P>
__global__ void __launch_bounds__(256) k_for_each_multi(const __grid_constant__ P pack, const __grid_constant__ MultiRanges r) {
  int k = 0;
  while (k + 1 < r.count && blockIdx.x >= r.blk_end[k]) k++;
  u32 i = (blockIdx.x - (k ? r.blk_end[k - 1] : 0u)) * blockDim.x + threadIdx.x;
  if (i < r.n[k]) pack.call(k, i);
}

// resident 256-thread blocks per SM each warp-synchronous stage is compiled for (register cap = 65536 / (256 * N)):
// these stages wait on dependent DRAM loads, so occupancy matters more than registers
template <class F> struct MinBlocks { static constexpr int value = 2; };
template <> struct MinBlocks<FGaObj> { static constexpr int value = 4; };
template <> struct MinBlocks<FR53Pair> { static constexpr int value = 6; };
template <> struct MinBlocks<FR53Prepare> { static constexpr int value = 6; };

__global__ void k_fill32(u32 *p, u32 v, size_t n) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  size_t stride = (size_t)gridDim.x * blockDim.x;
  for (; i < n; i += stride) p[i] = v;
}

// ---- exclusive scan (u32): per-tile reduce, single-block scan of tile sums, per-tile scan + offset
constexpr int SCAN_THREADS = 256;
constexpr int SCAN_ITEMS = 8;
constexpr int SCAN_TILE = SCAN_THREADS * SCAN_ITEMS;

__device__ __forceinline__ u32 warp_incl_scan(u32 v) {
  const unsigned lane = threadIdx.x & 31;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    u32 t = __shfl_up_sync(0xffffffffu, v, d);
    if (lane >= (unsigned)d) v += t;
  }
  return v;
}
// exclusive scan of one value per thread across the block; returns the exclusive prefix, *total = block sum
__device__ __forceinline__ u32 block_excl_scan(u32 v, u32 *total) {
  __shared__ u32 wsum[SCAN_THREADS / 32];
  __shared__ u32 wtot;
  const unsigned lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  u32 inc = warp_incl_scan(v);
  if (lane == 31) wsum[w] = inc;
  __syncthreads();
  if (w == 0) {
    u32 s = lane < SCAN_THREADS / 32 ? wsum[lane] : 0;
    u32 si = warp_incl_scan(s);
    if (lane < SCAN_THREADS / 32) wsum[lane] = si - s;
    if (lane == SCAN_THREADS / 32 - 1) wtot = si;
  }
  __syncthreads();
  u32 r = wsum[w] + inc - v;
  *total = wtot;
  __syncthreads();
  return r;
}

// Single-pass chained scan with decoupled look-back.  Tiles take a ticket (so a tile only ever waits on tiles that
// already run or ran), publish their aggregate, then their inclusive prefix; a tile's exclusive prefix is the sum
// of its predecessors' aggregates back to the first published inclusive prefix.
// state word: bits 62..63 = 0 empty, 1 aggregate, 2 inclusive prefix; low 32 bits = value.
__global__ void __launch_bounds__(SCAN_THREADS) k_scan_lookback(u32 *data, u32 n, unsigned long long *state, u32 *ticket) {
  __shared__ u32 s_tile, s_excl;
  if (threadIdx.x == 0) s_tile = atomicAdd(ticket, 1u);
  __syncthreads();
  const u32 tile = s_tile;
  const u32 base = tile * SCAN_TILE + threadIdx.x * SCAN_ITEMS;
  u32 v[SCAN_ITEMS];
  if (base + SCAN_ITEMS <= n) {
    const uint4 *q = reinterpret_cast<const uint4 *>(data + base);
    uint4 a = q[0], b = q[1];
    v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w;
    v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
  } else {
#pragma unroll
    for (int k = 0; k < SCAN_ITEMS; k++) v[k] = base + k < n ? data[base + k] : 0;
  }
  u32 s = 0;
#pragma unroll
  for (int k = 0; k < SCAN_ITEMS; k++) s += v[k];
  u32 total;
  u32 ex = block_excl_scan(s, &total);
  if (threadIdx.x < 32) {  // warp 0 looks back over 32 predecessors per step
    volatile unsigned long long *st = state;
    const unsigned lane = threadIdx.x;
    if (tile == 0) {
      if (lane == 0) {
        st[0] = (2ull << 62) | total;
        s_excl = 0;
      }
    } else {
      if (lane == 0) {
        st[tile] = (1ull << 62) | total;
        __threadfence();
      }
      u32 excl = 0;
      for (long long p = (long long)tile - 1;; p -= 32) {
        long long idx = p - (long long)lane;
        unsigned long long w = 2ull << 62;  // before tile 0: an inclusive prefix of 0
        if (idx >= 0) {
          do {
            w = st[idx];
          } while ((w >> 62) == 0);
        }
        unsigned pm = __ballot_sync(0xffffffffu, (w >> 62) == 2);
        int first = __ffs(pm) - 1;  // nearest predecessor that already knows its inclusive prefix
        u32 val = (first < 0 || (int)lane <= first) ? (u32)w : 0u;
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) val += __shfl_down_sync(0xffffffffu, val, off);
        excl += val;  // meaningful in lane 0
        if (first >= 0) break;
      }
      if (lane == 0) {
        st[tile] = (2ull << 62) | (u32)(excl + total);
        s_excl = excl;
      }
    }
  }
  __syncthreads();
  ex += s_excl;
  if (base + SCAN_ITEMS <= n) {
    uint4 a, b;
    a.x = ex; ex += v[0];
    a.y = ex; ex += v[1];
    a.z = ex; ex += v[2];
    a.w = ex; ex += v[3];
    b.x = ex; ex += v[4];
    b.y = ex; ex += v[5];
    b.z = ex; ex += v[6];
    b.w = ex;
    uint4 *q = reinterpret_cast<uint4 *>(data + base);
    q[0] = a;
    q[1] = b;
  } else {
#pragma unroll
    for (int k = 0; k < SCAN_ITEMS; k++) {
      if (base + k < n) data[base + k] = ex;
      ex += v[k];
    }
  }
}

// ---- stable LSD radix sort of (u32 key, u32 value) pairs, 8 bits per pass.
// Tile = 256 threads x 8 items; inside a tile item order is (warp, round, lane) = ascending index, and the
// per-digit rank is built with match_any so equal keys keep their input order.
constexpr int RS_THREADS = 256;
constexpr int RS_ITEMS = 8;
constexpr int RS_TILE = RS_THREADS * RS_ITEMS;
constexpr int RS_WARPS = RS_THREADS / 32;

__global__ void __launch_bounds__(RS_THREADS) k_radix_hist(const u32 *keys, u32 n, int shift, u32 *hist /* [256][ntiles] */, u32 ntiles) {
  __shared__ u32 h[256];
  h[threadIdx.x] = 0;
  __syncthreads();
  u32 base = blockIdx.x * RS_TILE;
#pragma unroll
  for (int k = 0; k < RS_ITEMS; k++) {
    u32 i = base + k * RS_THREADS + threadIdx.x;
    if (i < n) atomicAdd(&h[(keys[i] >> shift) & 255u], 1u);
  }
  __syncthreads();
  hist[(size_t)threadIdx.x * ntiles + blockIdx.x] = h[threadIdx.x];
}

__global__ void __launch_bounds__(RS_THREADS) k_radix_scatter(const u32 *keys, const u32 *vals, u32 *keys_out, u32 *vals_out, u32 n, int shift,
                                                              const u32 *hist_scanned, u32 ntiles) {
  __shared__ u32 wcnt[RS_WARPS][256];
  __shared__ u32 dbase[256];
  const unsigned lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  for (int k = threadIdx.x; k < RS_WARPS * 256; k += RS_THREADS) (&wcnt[0][0])[k] = 0;
  dbase[threadIdx.x] = hist_scanned[(size_t)threadIdx.x * ntiles + blockIdx.x];
  __syncthreads();
  const u32 wbase = blockIdx.x * RS_TILE + w * (32 * RS_ITEMS);
  u32 key[RS_ITEMS], val[RS_ITEMS], rank[RS_ITEMS];
#pragma unroll
  for (int r = 0; r < RS_ITEMS; r++) {
    u32 i = wbase + r * 32 + lane;
    bool ok = i < n;
    key[r] = ok ? keys[i] : 0;
    val[r] = ok ? vals[i] : 0;
    u32 d = ok ? ((key[r] >> shift) & 255u) : 256u;  // 256 = out-of-range items group together and are dropped
    unsigned peers = __match_any_sync(0xffffffffu, d);
    unsigned leader = __ffs(peers) - 1;
    u32 before = __popc(peers & ((1u << lane) - 1));
    u32 prev = 0;
    if (lane == leader && d < 256u) {
      prev = wcnt[w][d];
      wcnt[w][d] = prev + __popc(peers);
    }
    prev = __shfl_sync(0xffffffffu, prev, leader);
    rank[r] = prev + before;
    __syncwarp();
  }
  __syncthreads();
  {  // exclusive prefix over warps for digit = threadIdx.x
    u32 run = 0;
#pragma unroll
    for (int ww = 0; ww < RS_WARPS; ww++) {
      u32 c = wcnt[ww][threadIdx.x];
      wcnt[ww][threadIdx.x] = run;
      run += c;
    }
  }
  __syncthreads();
#pragma unroll
  for (int r = 0; r < RS_ITEMS; r++) {
    u32 i = wbase + r * 32 + lane;
    if (i < n) {
      u32 d = (key[r] >> shift) & 255u;
      u32 dst = dbase[d] + wcnt[w][d] + rank[r];
      keys_out[dst] = key[r];
      vals_out[dst] = val[r];
    }
  }
}

// ------------------------------------------------------------------ snapshot validation on the device
//
// Every string reference must stay inside its slab, every CSR must be monotone and closed, enums in range, and the object
// key layout rule must hold.  The checks run as tiny streaming kernels over the freshly copied tables (no host pass that
// would compete with the PCIe copy for memory bandwidth); the first failing check id lands in a flag the load reads back
// BEFORE any pipeline kernel can see the tables.
struct FValStr {
  const gar_str *col;
  u64 slab_len;
  u32 id;
  u32 *flag;
  __device__ void operator()(u32 i) const {
    gar_str r = col[i];
    if (GAR_STR_OFF(r) + GAR_STR_LEN(r) > slab_len) atomicMin(flag, id);
  }
};
struct FValCsr {
  const u32 *b;
  u32 nparents, nchildren, id;
  u32 *flag;
  __device__ void operator()(u32 i) const {  // i in [0, nparents]
    bool bad = (i == 0 && b[0] != 0) || (i < nparents && b[i + 1] < b[i]) || (i == nparents && b[nparents] != nchildren);
    if (bad) atomicMin(flag, id);
  }
};
struct FValObj {
  gar_objects o;
  u32 id_kind, id_key, id_icls;
  u32 *flag;
  __device__ void operator()(u32 i) const {
    if (o.obj_kind[i] > GAR_KIND_INGRESS || o.obj_spec_type[i] > GAR_SVC_EXTERNALNAME) atomicMin(flag, id_kind);
    u64 sep = GAR_STR_OFF(o.obj_ns[i]) + GAR_STR_LEN(o.obj_ns[i]);
    if (GAR_STR_OFF(o.obj_name[i]) != sep + 1 || sep >= o.slab_len || o.slab[sep] != '/') atomicMin(flag, id_key);
    // obj_ingress_class is meaningful only where the flag says so (garecon.h): other rows may hold anything
    if (o.obj_flags[i] & GAR_OBJ_HAS_INGRESS_CLASS) {
      gar_str r = o.obj_ingress_class[i];
      if (GAR_STR_OFF(r) + GAR_STR_LEN(r) > o.slab_len) atomicMin(flag, id_icls);
    }
  }
};
struct FValEnum {
  const u8 *col;
  u32 max_value, id;
  u32 *flag;
  __device__ void operator()(u32 i) const {
    if (col[i] > max_value) atomicMin(flag, id);
  }
};

// ------------------------------------------------------------------ engine

struct DBuf {
  void *p = nullptr;
  size_t cap = 0;
};

struct HostResult {  // pinned host buffers of one change set
  DBuf status_ga, status_r53, derived, ops, tok_code, tok_name, tok_region, dport_begin, dports, obj_gid;
};

#define CK(call)                                                                                             \
  do {                                                                                                       \
    cudaError_t _e = (call);                                                                                 \
    if (_e != cudaSuccess) {                                                                                 \
      char _b[512];                                                                                          \
      snprintf(_b, sizeof(_b), "%s failed: %s (%s:%d)", #call, cudaGetErrorString(_e), __FILE__, __LINE__); \
      throw CudaError{std::string(_b)};                                                                      \
    }                                                                                                        \
  } while (0)

struct CudaError {
  std::string msg;
};
struct InvalidError {
  std::string msg;
};
struct StateError {
  std::string msg;
};

static std::string g_create_error = "";

// Peer push (sharded mode, gar_shard_pack_peers): finished level groups of the staged blobs go to the other GPUs' receive arenas
// over NVLink as 16-byte coalesced stores, one grid row per destination.  Runs on a high-priority stream beside the pack
// kernels of the later levels.  (Measured at 8 GPUs, 2.6 GB to 7 peers per rank: copy engines 340 GB/s aggregate, last byte at
// 7.8 ms; this kernel: last byte 0.2 ms after the last pack kernel, at 6.8 ms; NCCL all-to-all after a separate pack: 7.9 ms.)
struct PushDesc {
  const uint4 *src[GAR_SHARD_MAX_RANKS];
  uint4 *dst[GAR_SHARD_MAX_RANKS];
  unsigned long long n16[GAR_SHARD_MAX_RANKS];
};
constexpr int PUSH_BLOCKS = 24, PUSH_THREADS = 512;
__global__ void __launch_bounds__(PUSH_THREADS) k_peer_push(const __grid_constant__ PushDesc d) {
  const uint4 *__restrict__ s = d.src[blockIdx.y];
  uint4 *__restrict__ t = d.dst[blockIdx.y];
  const unsigned long long n = d.n16[blockIdx.y], stride = (unsigned long long)gridDim.x * blockDim.x;
  unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
  for (; i + 3 * stride < n; i += 4 * stride) {
    uint4 a = __ldcs(s + i), b = __ldcs(s + i + stride), c = __ldcs(s + i + 2 * stride), e = __ldcs(s + i + 3 * stride);
    t[i] = a;
    t[i + stride] = b;
    t[i + 2 * stride] = c;
    t[i + 3 * stride] = e;
  }
  for (; i < n; i += stride) t[i] = __ldcs(s + i);
}

struct gar_engine {
  int device = 0;
  std::string cluster;
  std::string err;
  std::mutex mu;
  cudaStream_t stream = nullptr;
  cudaEvent_t ev[6] = {};
  bool loaded = false, attached = false;
  DevTables T{};
  std::vector<DBuf> in;        // device copies of the input arrays (copy mode)
  size_t in_used = 0;
  DBuf cluster_dev;
  DBuf slot[S_NSLOTS];
  DBuf d_status_ga, d_status_r53, d_derived, d_ops, d_tok_code, d_tok_name, d_tok_region, d_dport_begin, d_dports, d_scan_tiles, d_hist;
  DBuf d_derived_keys, d_key_rows, d_del_kind, d_del_key, d_del_slab;  // incremental mode
  DBuf d_egb[8];                                                      // EndpointGroupBinding tables
  DBuf d_valid;                                                       // validation flag
  Pipeline<gar_engine> *pipe = nullptr;  // lives as long as the loaded snapshot: keeps digests + indexes resident
  // sharded mode (gar_shard.h)
  Sharder<gar_engine> *sharder = nullptr;
  DevTables slice{};          // the loaded slice (T switches to the home sub-snapshot after the second unpack)
  bool shard_home = false;    // T is a home sub-snapshot: results are translated to global rows
  int shard_round = 0;        // last completed step: 1 routed1, 2 unpacked1, 3 routed2, 4 unpacked2
  u32 shard_launches = 0;     // kernels of the exchange steps since the last diff
  bool shard_reported = true; // stage marks of the exchange steps already folded into a diff's timings
  std::vector<DBuf> arena[3];
  size_t arena_used[3] = {0, 0, 0};
  void *shard_alloc(int a, size_t bytes) {
    if (arena_used[a] >= arena[a].size()) arena[a].emplace_back();
    return dev_ensure(arena[a][arena_used[a]++], bytes + 32);
  }
  void shard_reset(int a) { arena_used[a] = 0; }
  void copy_bytes(void *dst, const void *src, size_t n) {
    if (n) CK(cudaMemcpyAsync(dst, src, n, cudaMemcpyDeviceToDevice, stream));
  }
  // peer-memory exchange: this rank's receive arenas (one per round) and the mapped arenas of the other ranks
  struct PeerHandle {  // what travels in GAR_SHARD_HANDLE_BYTES
    u64 magic, pid, ptr, cap;
    cudaIpcMemHandle_t ipc;
  };
  static_assert(sizeof(PeerHandle) <= GAR_SHARD_HANDLE_BYTES, "handle does not fit");
  DBuf peer_arena[2];
  u8 *peer_ptr[2][GAR_SHARD_MAX_RANKS] = {};
  PeerHandle peer_seen[2][GAR_SHARD_MAX_RANKS] = {};
  bool peer_mapped[2][GAR_SHARD_MAX_RANKS] = {};
  // staged transfer: the blobs for the other ranks are packed into `peer_stage` and pushed to their arenas by k_peer_push,
  // level group by level group while the later levels still pack
  DBuf peer_stage;
  cudaStream_t peer_push_stream = nullptr;  // high priority: its blocks are placed before the pack kernels' next ones
  std::vector<cudaEvent_t> peer_ev;
  void peers_close() {
    for (int r = 0; r < 2; r++)
      for (int k = 0; k < GAR_SHARD_MAX_RANKS; k++) {
        if (peer_mapped[r][k]) cudaIpcCloseMemHandle(peer_ptr[r][k]);
        peer_mapped[r][k] = false;
        peer_ptr[r][k] = nullptr;
        peer_seen[r][k] = PeerHandle{};
      }
  }
  std::vector<HostResult *> free_results;
  float ms_h2d = 0;
  u32 launches = 0;
  u64 input_bytes = 0;  // slabs + fixed-width columns, each once
  // stage timing (GAR_FLAG_STAGE_TIMING)
  bool timing = false;
  bool reprepare = false;  // GAR_FLAG_REPREPARE
  bool no_orphans = false, allow_empty_cache = false;  // GAR_FLAG_NO_ORPHANS, GAR_FLAG_ALLOW_EMPTY_CACHE
  struct Mark {
    const char *name;
    cudaEvent_t a, b;
    u32 launches;
  };
  std::vector<Mark> marks;
  std::vector<cudaEvent_t> event_pool;
  size_t events_used = 0;
  int stage_depth = 0;
  u32 stage_launch0 = 0;
  std::vector<gar_stage_timing> last_timings;
  u64 last_counters[GAR_CTR_N] = {};
  cudaEvent_t new_event() {
    if (events_used == event_pool.size()) {
      cudaEvent_t ev;
      CK(cudaEventCreate(&ev));
      event_pool.push_back(ev);
    }
    return event_pool[events_used++];
  }
  void stage_begin(const char *name) {
    if (!timing || stage_depth++ > 0) return;
    Mark m{name, new_event(), new_event(), 0};
    CK(cudaEventRecord(m.a, stream));
    stage_launch0 = launches;
    marks.push_back(m);
  }
  void stage_end() {
    if (!timing || --stage_depth > 0) return;
    marks.back().launches = launches - stage_launch0;
    CK(cudaEventRecord(marks.back().b, stream));
  }

  // ---- memory
  void *dev_ensure(DBuf &b, size_t bytes) {
    bytes = (bytes + 255) & ~(size_t)255;
    if (b.cap < bytes) {
      if (capturing) throw CudaError{"internal: a buffer grew while a launch sequence was being recorded"};
      graph_drop();  // recorded launches hold the old pointer
      if (b.p) CK(cudaFree(b.p));
      b.p = nullptr;
      b.cap = 0;
      size_t want = bytes + bytes / 4;
      CK(cudaMalloc(&b.p, want));
      b.cap = want;
    }
    return b.p;
  }
  void *pin_ensure(DBuf &b, size_t bytes) {
    if (bytes < 64) bytes = 64;
    if (b.cap < bytes) {
      if (b.p) CK(cudaFreeHost(b.p));
      b.p = nullptr;
      b.cap = 0;
      size_t want = bytes + bytes / 4;
      CK(cudaMallocHost(&b.p, want));
      b.cap = want;
    }
    return b.p;
  }

  // ---- Backend interface (gar_pipeline.h)
  template <class F>
  void for_each(const char *name, u32 n, const F &f) {
    if (!n) return;
    stage_begin(name);
    k_for_each<F><<<(n + 255) / 256, 256, 0, stream>>>(f, n);
    launches++;
    stage_end();
  }
  template <class F>
  void for_each_warp(const char *name, u32 n, const F &f) {
    if (!n) return;
    stage_begin(name);
    k_for_each_warp<F, MinBlocks<F>::value><<<(n + 255) / 256, 256, 0, stream>>>(f, n);
    launches++;
    stage_end();
  }
  // ---- launch-sequence caching.  A full diff of an unchanged snapshot issues exactly the same launches with the same arguments
  // every time (all sizes that only the device knows live in capacity-sized buffers): the second such diff is recorded into
  // a CUDA graph, later ones replay it — one graph launch instead of ~35 kernel launches and memsets (what a 10^5-object diff
  // is bound by).  Anything that changes the sequence (new snapshot, a capacity that grew, stage timing) drops the graph.
  // capacities a previous snapshot's diffs settled on: the next snapshot of the same controller is almost always the same shape,
  // so its first diff starts with buffers that fit (no grow-and-rerun on every load)
  u32 hint_dport_cap = 0, hint_pair_cap = 0;
  u64 hint_ops_cap = 0;
  cudaGraphExec_t graph_exec = nullptr;
  u64 graph_sig = 0, seen_sig = 0;
  u32 graph_launches = 0, capture_launch0 = 0;
  bool capturing = false;
  void graph_drop() {
    if (graph_exec) cudaGraphExecDestroy(graph_exec);
    graph_exec = nullptr;
    graph_sig = seen_sig = 0;
  }
  int graph_begin(u64 sig) {
    if (timing) return 0;
    if (graph_exec && graph_sig == sig) {
      CK(cudaGraphLaunch(graph_exec, stream));
      launches += graph_launches;
      return 2;
    }
    if (seen_sig != sig) {  // first diff with this shape: run it eagerly (buffers get their sizes), remember the shape
      graph_drop();
      seen_sig = sig;
      return 0;
    }
    graph_drop();
    seen_sig = sig;
    CK(cudaStreamBeginCapture(stream, cudaStreamCaptureModeThreadLocal));
    capturing = true;
    capture_launch0 = launches;
    return 1;
  }
  void graph_end() {
    if (!capturing) return;
    capturing = false;
    cudaGraph_t g = nullptr;
    CK(cudaStreamEndCapture(stream, &g));
    cudaError_t ie = cudaGraphInstantiate(&graph_exec, g, 0);
    cudaGraphDestroy(g);
    if (ie != cudaSuccess) {
      graph_exec = nullptr;
      throw CudaError{std::string("cudaGraphInstantiate failed: ") + cudaGetErrorString(ie)};
    }
    graph_sig = seen_sig;
    graph_launches = launches - capture_launch0;
    CK(cudaGraphLaunch(graph_exec, stream));
  }
  void for_each_staged(const char *name, u32 n, const FTokenise &f) {
    if (!n) return;
    stage_begin(name);
    k_tokenise_staged<<<(n + 255) / 256, 256, 0, stream>>>(f, n);
    launches++;
    stage_end();
  }
  template <class F>
  void for_each_dyn(const char *name, const u32 *n_dev, u32 cap, const F &f) {
    if (!cap) return;
    stage_begin(name);
    k_for_each_dyn<F><<<(cap + 255) / 256, 256, 0, stream>>>(f, n_dev, cap);
    launches++;
    stage_end();
  }
  template <class F>
  void for_each_warp_dyn(const char *name, const u32 *n_dev, u32 cap, const F &f) {
    if (!cap) return;
    stage_begin(name);
    k_for_each_warp_dyn<F, MinBlocks<F>::value><<<(cap + 255) / 256, 256, 0, stream>>>(f, n_dev, cap);
    launches++;
    stage_end();
  }
  template <class... Fs>
  void for_each_multi(const char *name, std::initializer_list<u32> ns, const Fs &...fs) {
    static_assert(sizeof...(Fs) <= MULTI_MAX, "too many functors for one fused launch");
    MultiRanges r{};
    u32 blocks = 0;
    for (u32 n : ns) {
      blocks += (n + 255) / 256;
      r.blk_end[r.count] = blocks;
      r.n[r.count] = n;
      r.count++;
    }
    if (!blocks) return;
    stage_begin(name);
    k_for_each_multi<FPack<Fs...>><<<blocks, 256, 0, stream>>>(FPack<Fs...>(fs...), r);
    launches++;
    stage_end();
  }
  void fill32(u32 *p, u32 v, size_t n) {
    if (!n) return;
    if (v == 0) {
      CK(cudaMemsetAsync(p, 0, n * 4, stream));
      return;
    }
    size_t blocks = (n + 255) / 256;
    if (blocks > 148 * 16) blocks = 148 * 16;
    k_fill32<<<(unsigned)blocks, 256, 0, stream>>>(p, v, n);
    launches++;
  }
  void copy32(u32 *dst, const u32 *src, size_t n) {
    if (n) CK(cudaMemcpyAsync(dst, src, n * 4, cudaMemcpyDeviceToDevice, stream));
  }
  void exclusive_scan(u32 *data, u32 n) {
    if (!n) return;
    stage_begin("exclusive_scan");
    u32 ntiles = (n + SCAN_TILE - 1) / SCAN_TILE;
    size_t sbytes = 8 * (size_t)(ntiles + 2);
    unsigned long long *state = (unsigned long long *)dev_ensure(d_scan_tiles, sbytes);
    CK(cudaMemsetAsync(state, 0, sbytes, stream));  // tile states + the ticket counter (last word)
    k_scan_lookback<<<ntiles, SCAN_THREADS, 0, stream>>>(data, n, state, (u32 *)(state + ntiles + 1));
    launches += 1;
    stage_end();
  }
  void sort_pairs(u32 *keys, u32 *vals, u32 *keys_alt, u32 *vals_alt, u32 n, int bits) {
    if (!n) return;
    stage_begin("radix_sort_pairs");
    u32 ntiles = (n + RS_TILE - 1) / RS_TILE;
    u32 *hist = (u32 *)dev_ensure(d_hist, 4 * (size_t)256 * ntiles + 16);
    u32 *ka = keys, *va = vals, *kb = keys_alt, *vb = vals_alt;
    int passes = (bits + 7) / 8;
    for (int p = 0; p < passes; p++) {
      k_radix_hist<<<ntiles, RS_THREADS, 0, stream>>>(ka, n, p * 8, hist, ntiles);
      launches++;
      exclusive_scan(hist, 256 * ntiles);
      k_radix_scatter<<<ntiles, RS_THREADS, 0, stream>>>(ka, va, kb, vb, n, p * 8, hist, ntiles);
      launches++;
      std::swap(ka, kb);
      std::swap(va, vb);
    }
    if (ka != keys) {  // odd number of passes: bring the result back
      CK(cudaMemcpyAsync(keys, ka, 4 * (size_t)n, cudaMemcpyDeviceToDevice, stream));
      CK(cudaMemcpyAsync(vals, va, 4 * (size_t)n, cudaMemcpyDeviceToDevice, stream));
    }
    stage_end();
  }
  void *ensure(int s, size_t bytes) { return dev_ensure(slot[s], bytes); }
  void download(void *dst, const void *src, size_t bytes) {
    CK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, stream));
    CK(cudaStreamSynchronize(stream));
  }
  // small read-backs that travel while later stages are queued (pinned staging + an event each)
  DBuf dl_pin[2];
  cudaEvent_t dl_ev[2] = {};
  void download_start(int id, const void *src, size_t bytes) {
    void *p = pin_ensure(dl_pin[id], 64);
    if (!dl_ev[id]) CK(cudaEventCreateWithFlags(&dl_ev[id], cudaEventDisableTiming));
    CK(cudaMemcpyAsync(p, src, bytes, cudaMemcpyDeviceToHost, stream));
    CK(cudaEventRecord(dl_ev[id], stream));
  }
  void download_wait(int id, void *dst, size_t bytes) {
    CK(cudaEventSynchronize(dl_ev[id]));
    memcpy(dst, dl_pin[id].p, bytes);
  }
  void *out_derived(u32 n) { return dev_ensure(d_derived, 4 * (size_t)(n + 1)); }
  void *out_derived_keys(u32 n) { return dev_ensure(d_derived_keys, 4 * (size_t)(n + 1)); }
  void *out_dport_begin(u32 n) { return dev_ensure(d_dport_begin, 4 * (size_t)(n + 2)); }
  void *out_tok_code(u32 n) { return dev_ensure(d_tok_code, (size_t)n + 1); }
  void *out_tok_name(u32 n) { return dev_ensure(d_tok_name, 8 * (size_t)(n + 1)); }
  void *out_tok_region(u32 n) { return dev_ensure(d_tok_region, 8 * (size_t)(n + 1)); }
  void *out_dports(u64 n) { return dev_ensure(d_dports, 4 * (size_t)(n + 1)); }
  void *out_status_ga(u32 n) { return dev_ensure(d_status_ga, 4 * (size_t)(n + 1)); }
  void *out_status_r53(u32 n) { return dev_ensure(d_status_r53, 4 * (size_t)(n + 1)); }
};

// ------------------------------------------------------------------ host-side checks of small tables (bindings) and of pointers

static void check_str_col(const char *name, const gar_str *col, size_t n, u64 slab_len) {
  if (n && !col) throw InvalidError{std::string(name) + " is NULL"};
  for (size_t i = 0; i < n; i++) {
    u64 off = GAR_STR_OFF(col[i]), len = GAR_STR_LEN(col[i]);
    if (off + len > slab_len) throw InvalidError{std::string(name) + ": string reference outside the slab"};
  }
}
static void check_csr(const char *name, const u32 *b, size_t nparents, size_t nchildren) {
  if (!b) throw InvalidError{std::string(name) + " is NULL"};
  if (b[0] != 0) throw InvalidError{std::string(name) + "[0] != 0"};
  for (size_t i = 0; i < nparents; i++)
    if (b[i + 1] < b[i]) throw InvalidError{std::string(name) + " is not monotone"};
  if (b[nparents] != nchildren) throw InvalidError{std::string(name) + " does not end at the child count"};
}
static void check_ptr(const char *name, const void *p, size_t n) {
  if (n && !p) throw InvalidError{std::string(name) + " is NULL"};
}

// bytes of the input tables, each array counted once (roofline numerator, DESIGN.md)
static u64 table_bytes(const gar_objects *o, const gar_actual *a) {
  u64 n = o->n_objects, b = 0;
  b += o->slab_len + a->slab_len;
  b += n * (3 + 8 * 3) + 4 * (n + 1) * 3;
  b += (u64)o->n_ann * 16 + (u64)o->n_lbi * 8 + (u64)o->n_ports * 12;
  b += (u64)a->n_lbs * (8 * 4 + 1);
  b += (u64)a->n_accels * (8 * 2 + 1) + 4 * ((u64)a->n_accels + 1) * 2;
  b += (u64)a->n_tags * 16;
  b += (u64)a->n_listeners * 1 + 4 * ((u64)a->n_listeners + 1) * 2;
  b += (u64)a->n_port_ranges * 4;
  b += 4 * ((u64)a->n_egs + 1);
  b += (u64)a->n_endpoints * 8;
  b += (u64)a->n_zones * 8 + 4 * ((u64)a->n_zones + 1);
  b += (u64)a->n_records * (8 + 1 + 1 + 8) + 4 * ((u64)a->n_records + 1);
  b += (u64)a->n_values * 8;
  return b;
}

// ------------------------------------------------------------------ load

static void validate_pointers(const gar_objects *o, const gar_actual *a) {
  size_t n = o->n_objects;
  check_ptr("obj_kind", o->obj_kind, n); check_ptr("obj_spec_type", o->obj_spec_type, n); check_ptr("obj_flags", o->obj_flags, n);
  check_ptr("obj_ns", o->obj_ns, n); check_ptr("obj_name", o->obj_name, n); check_ptr("obj_ingress_class", o->obj_ingress_class, n);
  check_ptr("obj_ann_begin", o->obj_ann_begin, 1); check_ptr("obj_lbi_begin", o->obj_lbi_begin, 1); check_ptr("obj_port_begin", o->obj_port_begin, 1);
  check_ptr("ann_key", o->ann_key, o->n_ann); check_ptr("ann_val", o->ann_val, o->n_ann); check_ptr("lbi_hostname", o->lbi_hostname, o->n_lbi);
  check_ptr("port_number", o->port_number, o->n_ports); check_ptr("port_proto", o->port_proto, o->n_ports); check_ptr("objects.slab", o->slab, o->slab_len);
  check_ptr("lb_region", a->lb_region, a->n_lbs); check_ptr("lb_name", a->lb_name, a->n_lbs); check_ptr("lb_dns", a->lb_dns, a->n_lbs);
  check_ptr("lb_arn", a->lb_arn, a->n_lbs); check_ptr("lb_state", a->lb_state, a->n_lbs);
  check_ptr("acc_name", a->acc_name, a->n_accels); check_ptr("acc_dns", a->acc_dns, a->n_accels); check_ptr("acc_enabled", a->acc_enabled, a->n_accels);
  check_ptr("acc_tag_begin", a->acc_tag_begin, 1); check_ptr("acc_lis_begin", a->acc_lis_begin, 1);
  check_ptr("tag_key", a->tag_key, a->n_tags); check_ptr("tag_val", a->tag_val, a->n_tags); check_ptr("lis_proto", a->lis_proto, a->n_listeners);
  check_ptr("lis_pr_begin", a->lis_pr_begin, 1); check_ptr("lis_eg_begin", a->lis_eg_begin, 1); check_ptr("pr_from", a->pr_from, a->n_port_ranges);
  check_ptr("eg_ep_begin", a->eg_ep_begin, 1); check_ptr("ep_id", a->ep_id, a->n_endpoints);
  check_ptr("zone_name", a->zone_name, a->n_zones); check_ptr("zone_rec_begin", a->zone_rec_begin, 1);
  check_ptr("rec_name", a->rec_name, a->n_records); check_ptr("rec_type", a->rec_type, a->n_records); check_ptr("rec_has_alias", a->rec_has_alias, a->n_records);
  check_ptr("rec_alias_dns", a->rec_alias_dns, a->n_records); check_ptr("rec_val_begin", a->rec_val_begin, 1);
  check_ptr("val_value", a->val_value, a->n_values); check_ptr("actual.slab", a->slab, a->slab_len);
}

// runs on e->stream after the copies; throws InvalidError naming the first failing check
static void device_validate(gar_engine *e) {
  const gar_objects &o = e->T.o;
  const gar_actual &a = e->T.a;
  u32 *flag = (u32 *)e->dev_ensure(e->d_valid, 64);
  CK(cudaMemsetAsync(flag, 0xFF, 4, e->stream));
  std::vector<const char *> names;
  auto str = [&](const char *name, const gar_str *col, u32 n, u64 slab_len) {
    names.push_back(name);
    e->for_each("validate", n, FValStr{col, slab_len, (u32)names.size() - 1, flag});
  };
  auto csr = [&](const char *name, const u32 *b, u32 nparents, u32 nchildren) {
    names.push_back(name);
    e->for_each("validate", nparents + 1, FValCsr{b, nparents, nchildren, (u32)names.size() - 1, flag});
  };
  const u32 n = o.n_objects;
  names.push_back("obj_kind / obj_spec_type out of range");
  names.push_back("objects layout rule violated: obj_ns and obj_name must be slices of one \"ns/name\" key string");
  auto en = [&](const char *name, const u8 *col, u32 cnt, u32 max_value) {
    names.push_back(name);
    e->for_each("validate", cnt, FValEnum{col, max_value, (u32)names.size() - 1, flag});
  };
  str("obj_ns", o.obj_ns, n, o.slab_len); str("obj_name", o.obj_name, n, o.slab_len);
  names.push_back("obj_ingress_class");
  e->for_each("validate", n, FValObj{o, 0, 1, (u32)names.size() - 1, flag});
  en("lb_state out of range", a.lb_state, a.n_lbs, GAR_LB_FAILED); en("lis_proto out of range", a.lis_proto, a.n_listeners, GAR_PROTO_UDP);
  en("rec_type out of range", a.rec_type, a.n_records, GAR_RR_AAAA);
  csr("obj_ann_begin", o.obj_ann_begin, n, o.n_ann); csr("obj_lbi_begin", o.obj_lbi_begin, n, o.n_lbi); csr("obj_port_begin", o.obj_port_begin, n, o.n_ports);
  str("ann_key", o.ann_key, o.n_ann, o.slab_len); str("ann_val", o.ann_val, o.n_ann, o.slab_len); str("lbi_hostname", o.lbi_hostname, o.n_lbi, o.slab_len);
  str("port_proto", o.port_proto, o.n_ports, o.slab_len);
  str("lb_region", a.lb_region, a.n_lbs, a.slab_len); str("lb_name", a.lb_name, a.n_lbs, a.slab_len); str("lb_dns", a.lb_dns, a.n_lbs, a.slab_len);
  str("lb_arn", a.lb_arn, a.n_lbs, a.slab_len); str("acc_name", a.acc_name, a.n_accels, a.slab_len); str("acc_dns", a.acc_dns, a.n_accels, a.slab_len);
  csr("acc_tag_begin", a.acc_tag_begin, a.n_accels, a.n_tags); csr("acc_lis_begin", a.acc_lis_begin, a.n_accels, a.n_listeners);
  str("tag_key", a.tag_key, a.n_tags, a.slab_len); str("tag_val", a.tag_val, a.n_tags, a.slab_len);
  csr("lis_pr_begin", a.lis_pr_begin, a.n_listeners, a.n_port_ranges); csr("lis_eg_begin", a.lis_eg_begin, a.n_listeners, a.n_egs);
  csr("eg_ep_begin", a.eg_ep_begin, a.n_egs, a.n_endpoints); str("ep_id", a.ep_id, a.n_endpoints, a.slab_len);
  str("zone_name", a.zone_name, a.n_zones, a.slab_len); csr("zone_rec_begin", a.zone_rec_begin, a.n_zones, a.n_records);
  str("rec_name", a.rec_name, a.n_records, a.slab_len); str("rec_alias_dns", a.rec_alias_dns, a.n_records, a.slab_len);
  csr("rec_val_begin", a.rec_val_begin, a.n_records, a.n_values); str("val_value", a.val_value, a.n_values, a.slab_len);
  u32 bad = 0xFFFFFFFFu;
  e->download(&bad, flag, 4);  // synchronises e->stream: copies and checks are complete
  if (bad != 0xFFFFFFFFu) {
    std::string nm = bad < names.size() ? names[bad] : "table";
    if (bad >= 2 && !strstr(nm.c_str(), "out of range"))
      nm += strstr(nm.c_str(), "_begin") ? ": CSR is not monotone, does not start at 0 or does not end at the child count" : ": string reference outside the slab";
    throw InvalidError{nm};
  }
}

template <class Tp>
static const Tp *upload(gar_engine *e, const Tp *host, size_t count, size_t pad_bytes = 0) {
  if (e->in_used >= e->in.size()) e->in.emplace_back();
  DBuf &b = e->in[e->in_used++];
  size_t bytes = count * sizeof(Tp);
  e->dev_ensure(b, bytes + pad_bytes + 16);
  if (bytes) CK(cudaMemcpyAsync(b.p, host, bytes, cudaMemcpyHostToDevice, e->stream));
  if (pad_bytes) CK(cudaMemsetAsync((char *)b.p + bytes, 0, pad_bytes, e->stream));
  return (const Tp *)b.p;
}

static void do_load(gar_engine *e, const gar_objects *o, const gar_actual *a) {
  if (!o || !a) throw InvalidError{"NULL table struct"};
  e->loaded = false;
  e->graph_drop();
  delete e->pipe;  // the prepared state belongs to the previous snapshot
  e->pipe = nullptr;
  validate_pointers(o, a);  // NULL checks before anything is copied; the contents are checked on the device, below
  CK(cudaSetDevice(e->device));
  e->in_used = 0;
  DevTables &T = e->T;
  CK(cudaEventRecord(e->ev[0], e->stream));
  T.o = *o;
  T.a = *a;
  size_t n = o->n_objects;
  T.o.obj_kind = upload(e, o->obj_kind, n);
  T.o.obj_spec_type = upload(e, o->obj_spec_type, n);
  T.o.obj_flags = upload(e, o->obj_flags, n);
  T.o.obj_ns = upload(e, o->obj_ns, n);
  T.o.obj_name = upload(e, o->obj_name, n);
  T.o.obj_ingress_class = upload(e, o->obj_ingress_class, n);
  T.o.obj_ann_begin = upload(e, o->obj_ann_begin, n + 1);
  T.o.obj_lbi_begin = upload(e, o->obj_lbi_begin, n + 1);
  T.o.obj_port_begin = upload(e, o->obj_port_begin, n + 1);
  T.o.ann_key = upload(e, o->ann_key, o->n_ann);
  T.o.ann_val = upload(e, o->ann_val, o->n_ann);
  T.o.lbi_hostname = upload(e, o->lbi_hostname, o->n_lbi);
  T.o.port_number = upload(e, o->port_number, o->n_ports);
  T.o.port_proto = upload(e, o->port_proto, o->n_ports);
  T.o.slab = upload(e, o->slab, o->slab_len, GAR_SLAB_PAD);
  T.a.lb_region = upload(e, a->lb_region, a->n_lbs);
  T.a.lb_name = upload(e, a->lb_name, a->n_lbs);
  T.a.lb_dns = upload(e, a->lb_dns, a->n_lbs);
  T.a.lb_arn = upload(e, a->lb_arn, a->n_lbs);
  T.a.lb_state = upload(e, a->lb_state, a->n_lbs);
  T.a.acc_name = upload(e, a->acc_name, a->n_accels);
  T.a.acc_dns = upload(e, a->acc_dns, a->n_accels);
  T.a.acc_enabled = upload(e, a->acc_enabled, a->n_accels);
  T.a.acc_tag_begin = upload(e, a->acc_tag_begin, (size_t)a->n_accels + 1);
  T.a.acc_lis_begin = upload(e, a->acc_lis_begin, (size_t)a->n_accels + 1);
  T.a.tag_key = upload(e, a->tag_key, a->n_tags);
  T.a.tag_val = upload(e, a->tag_val, a->n_tags);
  T.a.lis_proto = upload(e, a->lis_proto, a->n_listeners);
  T.a.lis_pr_begin = upload(e, a->lis_pr_begin, (size_t)a->n_listeners + 1);
  T.a.lis_eg_begin = upload(e, a->lis_eg_begin, (size_t)a->n_listeners + 1);
  T.a.pr_from = upload(e, a->pr_from, a->n_port_ranges);
  T.a.eg_ep_begin = upload(e, a->eg_ep_begin, (size_t)a->n_egs + 1);
  T.a.ep_id = upload(e, a->ep_id, a->n_endpoints);
  T.a.zone_name = upload(e, a->zone_name, a->n_zones);
  T.a.zone_rec_begin = upload(e, a->zone_rec_begin, (size_t)a->n_zones + 1);
  T.a.rec_name = upload(e, a->rec_name, a->n_records);
  T.a.rec_type = upload(e, a->rec_type, a->n_records);
  T.a.rec_has_alias = upload(e, a->rec_has_alias, a->n_records);
  T.a.rec_alias_dns = upload(e, a->rec_alias_dns, a->n_records);
  T.a.rec_val_begin = upload(e, a->rec_val_begin, (size_t)a->n_records + 1);
  T.a.val_value = upload(e, a->val_value, a->n_values);
  T.a.slab = upload(e, a->slab, a->slab_len, GAR_SLAB_PAD);
  CK(cudaEventRecord(e->ev[1], e->stream));
  device_validate(e);
  CK(cudaEventElapsedTime(&e->ms_h2d, e->ev[0], e->ev[1]));  // device_validate synchronised: the caller may free its buffers
  e->input_bytes = table_bytes(o, a);
  e->loaded = true;
  e->attached = false;
  e->slice = e->T;
  e->shard_home = false;
  e->shard_round = 0;
}

// ------------------------------------------------------------------ diff

static void do_diff(gar_engine *e, gar_changeset *out, bool to_host, const gar_keyset *ks = nullptr, const gar_bindings *bd = nullptr) {
  if (!e->loaded) throw InvalidError{"no snapshot loaded"};
  CK(cudaSetDevice(e->device));
  memset(out, 0, sizeof(*out));
  e->launches = e->shard_home ? e->shard_launches : 0;  // a sharded step counts its routing / packing / merging kernels too
  e->shard_launches = 0;
  if (!e->shard_home || e->shard_reported) {
    e->marks.clear();
    e->events_used = 0;
  }
  e->shard_reported = true;
  e->stage_depth = 0;
  if (e->shard_home && (ks || bd)) throw InvalidError{"incremental / binding diffs are not available on a sharded sub-snapshot"};
  if (e->shard_home && e->shard_round != 4)
    throw StateError{"a new exchange has started: the previous sub-snapshot's strings live in receive buffers that are being refilled; "
                     "finish both rounds (gar_shard_unpack(.., 2, ..)) before the next diff"};
  if (!e->pipe) {
    e->graph_drop();  // recorded launches belong to the previous pipeline's buffers and tables
    e->pipe = new Pipeline<gar_engine>(*e, e->T);
    if (const char *tc = getenv("GAR_TINY_CAPS")) e->pipe->tiny_caps = tc[0] == '1';
    if (!e->pipe->tiny_caps) {
      e->pipe->dport_cap = e->hint_dport_cap;
      e->pipe->pair_cap = e->hint_pair_cap;
      e->pipe->ops_cap = e->hint_ops_cap;
    }
    if (e->shard_home) {
      e->pipe->acc_guest_from = e->sharder->guest_from;
      e->pipe->sharded = 1;
    }
  }
  Pipeline<gar_engine> &P = *e->pipe;
  P.orphan_sweep = !e->no_orphans;
  P.allow_empty_cache = e->allow_empty_cache;
  if (e->reprepare) P.prepared = false;
  DiffCounts dc{};
  auto ops_alloc = [&](u64 nops) { return e->dev_ensure(e->d_ops, sizeof(gar_op) * (size_t)(nops + 1)); };
  CK(cudaEventRecord(e->ev[2], e->stream));
  int rc;
  u32 n_out = e->T.o.n_objects;
  if (bd) {
    // EndpointGroupBinding set-diff: validate and upload the (small) binding tables
    const gar_bindings &b = *bd;
    size_t nb = b.n_bindings;
    if (nb && (!b.egb_flags || !b.egb_ref_kind)) throw InvalidError{"NULL binding columns"};
    check_str_col("egb_ref_key", b.egb_ref_key, nb, b.slab_len);
    check_str_col("egb_eg_arn", b.egb_eg_arn, nb, b.slab_len);
    check_csr("egb_ep_begin", b.egb_ep_begin, nb, b.n_endpoint_ids);
    check_str_col("ep_id", b.ep_id, b.n_endpoint_ids, b.slab_len);
    check_str_col("known_eg_arn", b.known_eg_arn, b.n_known_egs, b.slab_len);
    for (size_t k = 0; k < nb; k++)
      if (b.egb_ref_kind[k] > GAR_EGB_REF_INGRESS) throw InvalidError{"egb_ref_kind out of range"};
    auto up = [&](DBuf &db, const void *src, size_t bytes, size_t pad) -> void * {
      void *p = e->dev_ensure(db, bytes + pad + 16);
      if (bytes) CK(cudaMemcpyAsync(p, src, bytes, cudaMemcpyHostToDevice, e->stream));
      if (pad) CK(cudaMemsetAsync((char *)p + bytes, 0, pad, e->stream));
      return p;
    };
    gar_bindings d = b;
    d.egb_flags = (const u8 *)up(e->d_egb[0], b.egb_flags, nb, 0);
    d.egb_ref_kind = (const u8 *)up(e->d_egb[1], b.egb_ref_kind, nb, 0);
    d.egb_ref_key = (const gar_str *)up(e->d_egb[2], b.egb_ref_key, 8 * nb, 0);
    d.egb_eg_arn = (const gar_str *)up(e->d_egb[3], b.egb_eg_arn, 8 * nb, 0);
    d.egb_ep_begin = (const u32 *)up(e->d_egb[4], b.egb_ep_begin, 4 * (nb + 1), 0);
    d.ep_id = (const gar_str *)up(e->d_egb[5], b.ep_id, 8 * (size_t)b.n_endpoint_ids, 0);
    d.known_eg_arn = (const gar_str *)up(e->d_egb[6], b.known_eg_arn, 8 * (size_t)b.n_known_egs, 0);
    d.slab = (const u8 *)up(e->d_egb[7], b.slab, b.slab_len, GAR_SLAB_PAD);
    CK(cudaStreamSynchronize(e->stream));
    n_out = b.n_bindings;
    rc = P.run_bindings(d, &dc, ops_alloc);
  } else if (!ks) {
    rc = P.run(&dc, ops_alloc);
  } else {
    // incremental mode: upload the key batch (rows + deleted keys)
    if ((ks->n_rows && !ks->rows) || (ks->n_deleted && (!ks->deleted_kind || !ks->deleted_key))) throw InvalidError{"NULL key set arrays"};
    for (u32 k = 0; k < ks->n_rows; k++)
      if (ks->rows[k] >= e->T.o.n_objects) throw InvalidError{"key set row out of range"};
    n_out = ks->n_rows;
    u32 *rows = (u32 *)e->dev_ensure(e->d_key_rows, 4 * (size_t)(ks->n_rows + 1));
    if (ks->n_rows) CK(cudaMemcpyAsync(rows, ks->rows, 4 * (size_t)ks->n_rows, cudaMemcpyHostToDevice, e->stream));
    std::vector<u8> slab;
    std::vector<gar_str> refs(ks->n_deleted);
    std::vector<u8> kinds(ks->n_deleted);
    for (u32 k = 0; k < ks->n_deleted; k++) {
      if (!ks->deleted_key[k] || ks->deleted_kind[k] > GAR_KIND_INGRESS) throw InvalidError{"bad deleted key"};
      size_t len = strlen(ks->deleted_key[k]);
      refs[k] = GAR_STR(slab.size(), len);
      slab.insert(slab.end(), ks->deleted_key[k], ks->deleted_key[k] + len);
      kinds[k] = ks->deleted_kind[k];
    }
    slab.resize(slab.size() + GAR_SLAB_PAD, 0);
    u8 *dslab = (u8 *)e->dev_ensure(e->d_del_slab, slab.size());
    u8 *dkind = (u8 *)e->dev_ensure(e->d_del_kind, ks->n_deleted + 1);
    gar_str *dkey = (gar_str *)e->dev_ensure(e->d_del_key, 8 * (size_t)(ks->n_deleted + 1));
    CK(cudaMemcpyAsync(dslab, slab.data(), slab.size(), cudaMemcpyHostToDevice, e->stream));
    if (ks->n_deleted) {
      CK(cudaMemcpyAsync(dkind, kinds.data(), ks->n_deleted, cudaMemcpyHostToDevice, e->stream));
      CK(cudaMemcpyAsync(dkey, refs.data(), 8 * (size_t)ks->n_deleted, cudaMemcpyHostToDevice, e->stream));
    }
    CK(cudaStreamSynchronize(e->stream));  // the staging vectors go out of scope
    rc = P.run_keys(rows, ks->n_rows, DelKeys{dkind, dkey, dslab}, ks->n_deleted, &dc, ops_alloc);
  }
  if (rc == GAR_OK && e->shard_home && dc.n_ops) e->for_each("shard_translate_ops", (u32)dc.n_ops, FShTranslateOps{(gar_op *)e->d_ops.p, e->sharder->gids});
  CK(cudaEventRecord(e->ev[3], e->stream));
  if (rc == GAR_E_INVALID) {
    throw InvalidError{"objects layout rule violated: obj_ns and obj_name must be slices of one \"ns/name\" key string"};
  }
  if (rc == GAR_REFUSE_EMPTY_CACHE) {
    throw StateError{"the object table is empty but this cluster still owns AWS resources: refusing to emit delete-everything orphan sections "
                     "(informer not synced?).  Set GAR_FLAG_ALLOW_EMPTY_CACHE if the cache really is empty, or GAR_FLAG_NO_ORPHANS"};
  }
  if (rc != GAR_OK) throw InvalidError{"the diff did not settle: an intermediate relation kept outgrowing its buffer"};
  const bool partial = ks || bd;
  const u32 n = n_out, nlbi = partial ? 0 : e->T.o.n_lbi;
  const DBuf &d_derived_src = ks ? e->d_derived_keys : e->d_derived;
  out->n_objects = n;
  out->n_ops = dc.n_ops;
  for (int k = 0; k <= GAR_N_SECTIONS; k++) out->section_begin[k] = dc.section_begin[k];
  out->n_lbi = nlbi;
  out->n_dports = dc.n_dports;
  if (to_host) {
    HostResult *h;
    if (!e->free_results.empty()) {
      h = e->free_results.back();
      e->free_results.pop_back();
    } else {
      h = new HostResult();
    }
    out->opaque = h;
    auto pull = [&](DBuf &hb, const DBuf &db, size_t bytes) -> void * {
      void *p = e->pin_ensure(hb, bytes);
      if (bytes) CK(cudaMemcpyAsync(p, db.p, bytes, cudaMemcpyDeviceToHost, e->stream));
      return p;
    };
    out->status_ga = (const u32 *)pull(h->status_ga, e->d_status_ga, 4 * (size_t)n);
    out->status_r53 = (const u32 *)pull(h->status_r53, e->d_status_r53, bd ? 0 : 4 * (size_t)n);
    out->derived = (const u32 *)pull(h->derived, d_derived_src, bd ? 0 : 4 * (size_t)n);
    out->ops = (const gar_op *)pull(h->ops, e->d_ops, sizeof(gar_op) * (size_t)dc.n_ops);
    out->tok_code = (const u8 *)pull(h->tok_code, e->d_tok_code, nlbi);
    out->tok_name = (const gar_str *)pull(h->tok_name, e->d_tok_name, 8 * (size_t)nlbi);
    out->tok_region = (const gar_str *)pull(h->tok_region, e->d_tok_region, 8 * (size_t)nlbi);
    out->dport_begin = (const u32 *)pull(h->dport_begin, e->d_dport_begin, partial ? 0 : 4 * (size_t)(n + 1));
    out->dports = (const i32 *)pull(h->dports, e->d_dports, 4 * (size_t)dc.n_dports);
    if (e->shard_home) {
      void *p = e->pin_ensure(h->obj_gid, 4 * (size_t)n);
      if (n) CK(cudaMemcpyAsync(p, e->sharder->gids.obj, 4 * (size_t)n, cudaMemcpyDeviceToHost, e->stream));
      out->obj_gid = (const u32 *)p;
    }
  } else {
    if (e->shard_home) out->obj_gid = e->sharder->gids.obj;
    out->status_ga = (const u32 *)e->d_status_ga.p;
    out->status_r53 = (const u32 *)e->d_status_r53.p;
    out->derived = (const u32 *)d_derived_src.p;
    out->ops = (const gar_op *)e->d_ops.p;
    out->tok_code = (const u8 *)e->d_tok_code.p;
    out->tok_name = (const gar_str *)e->d_tok_name.p;
    out->tok_region = (const gar_str *)e->d_tok_region.p;
    out->dport_begin = (const u32 *)e->d_dport_begin.p;
    out->dports = (const i32 *)e->d_dports.p;
  }
  CK(cudaEventRecord(e->ev[4], e->stream));
  CK(cudaStreamSynchronize(e->stream));
  CK(cudaGetLastError());
  CK(cudaEventElapsedTime(&out->ms_kernels, e->ev[2], e->ev[3]));
  CK(cudaEventElapsedTime(&out->ms_d2h, e->ev[3], e->ev[4]));
  out->ms_h2d = e->ms_h2d;
  out->kernel_launches = e->launches;
  if (!ks && !bd) {  // remember what a full diff of this shape needs
    e->hint_dport_cap = P.dport_cap;
    e->hint_pair_cap = P.pair_cap;
    e->hint_ops_cap = P.ops_cap;
  }
  e->last_counters[GAR_CTR_R53_PAIRS] = P.n_pairs;
  e->last_counters[GAR_CTR_DPORTS] = dc.n_dports;
  e->last_timings.clear();
  for (auto &m : e->marks) {
    float ms = 0;
    CK(cudaEventElapsedTime(&ms, m.a, m.b));
    bool found = false;
    for (auto &t : e->last_timings)
      if (!strcmp(t.name, m.name)) {
        t.ms += ms;
        t.launches += m.launches;
        found = true;
      }
    if (!found) e->last_timings.push_back(gar_stage_timing{m.name, ms, m.launches, 0});
  }
}

// ------------------------------------------------------------------ C ABI

template <class Fn>
static int guarded(gar_engine *e, Fn fn) {
  if (!e) return GAR_E_INVALID;
  std::lock_guard<std::mutex> lk(e->mu);
  try {
    fn();
    e->err.clear();
    return GAR_OK;
  } catch (const CudaError &ce) {
    e->err = ce.msg;
    if (e->capturing) {  // abandon a half-recorded launch sequence
      cudaGraph_t g = nullptr;
      cudaStreamEndCapture(e->stream, &g);
      if (g) cudaGraphDestroy(g);
      e->capturing = false;
    }
    e->graph_drop();
    cudaGetLastError();
    return GAR_E_CUDA;
  } catch (const InvalidError &ie) {
    e->err = ie.msg;
    return GAR_E_INVALID;
  } catch (const StateError &se) {
    e->err = se.msg;
    return GAR_E_STATE;
  } catch (const std::bad_alloc &) {
    e->err = "out of host memory";
    return GAR_E_NOMEM;
  }
}

extern "C" {

int gar_engine_create(const gar_config *cfg, gar_engine **out) {
  if (out) *out = nullptr;
  if (!cfg || !out || cfg->abi_version != GAR_ABI_VERSION) {
    g_create_error = "bad config or ABI version mismatch";
    return GAR_E_INVALID;
  }
  int ndev = 0;
  cudaError_t ce = cudaGetDeviceCount(&ndev);
  if (ce != cudaSuccess || ndev == 0 || cfg->device < 0 || cfg->device >= ndev) {
    g_create_error = std::string("no usable CUDA device: ") + (ce != cudaSuccess ? cudaGetErrorString(ce) : "device ordinal out of range");
    cudaGetLastError();
    return GAR_E_NO_DEVICE;
  }
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, cfg->device) != cudaSuccess || prop.major != 10) {
    g_create_error = "device is not sm_100 (this library ships sm_100a code only)";
    cudaGetLastError();
    return GAR_E_NO_DEVICE;
  }
  gar_engine *e = new gar_engine();
  e->device = cfg->device;
  e->cluster = cfg->cluster_name ? cfg->cluster_name : "";
  e->timing = (cfg->flags & GAR_FLAG_STAGE_TIMING) != 0;
  e->reprepare = (cfg->flags & GAR_FLAG_REPREPARE) != 0;
  e->no_orphans = (cfg->flags & GAR_FLAG_NO_ORPHANS) != 0;
  e->allow_empty_cache = (cfg->flags & GAR_FLAG_ALLOW_EMPTY_CACHE) != 0;
  try {
    CK(cudaSetDevice(e->device));
    CK(cudaStreamCreateWithFlags(&e->stream, cudaStreamNonBlocking));
    for (auto &ev : e->ev) CK(cudaEventCreate(&ev));
    e->dev_ensure(e->cluster_dev, e->cluster.size() + GAR_SLAB_PAD);
    CK(cudaMemsetAsync(e->cluster_dev.p, 0, e->cluster.size() + GAR_SLAB_PAD, e->stream));
    if (!e->cluster.empty()) CK(cudaMemcpyAsync(e->cluster_dev.p, e->cluster.data(), e->cluster.size(), cudaMemcpyHostToDevice, e->stream));
    CK(cudaStreamSynchronize(e->stream));
  } catch (const CudaError &err) {
    g_create_error = err.msg;
    delete e;
    return GAR_E_CUDA;
  }
  *out = e;
  return GAR_OK;
}

void gar_engine_destroy(gar_engine *e) {
  if (!e) return;
  cudaSetDevice(e->device);
  if (e->stream) cudaStreamSynchronize(e->stream);
  e->graph_drop();
  for (auto &b : e->in) cudaFree(b.p);
  for (auto &b : e->slot) cudaFree(b.p);
  delete e->pipe;
  delete e->sharder;
  e->peers_close();
  for (auto &b : e->peer_arena) cudaFree(b.p);
  cudaFree(e->peer_stage.p);
  if (e->peer_push_stream) cudaStreamDestroy(e->peer_push_stream);
  for (auto ev : e->peer_ev) cudaEventDestroy(ev);
  for (auto &ar : e->arena)
    for (auto &b : ar) cudaFree(b.p);
  for (DBuf *b : {&e->d_derived_keys, &e->d_key_rows, &e->d_del_kind, &e->d_del_key, &e->d_del_slab}) cudaFree(b->p);
  for (auto &b : e->d_egb) cudaFree(b.p);
  cudaFree(e->d_valid.p);
  for (int k = 0; k < 2; k++) {
    if (e->dl_pin[k].p) cudaFreeHost(e->dl_pin[k].p);
    if (e->dl_ev[k]) cudaEventDestroy(e->dl_ev[k]);
  }
  for (DBuf *b : {&e->cluster_dev, &e->d_status_ga, &e->d_status_r53, &e->d_derived, &e->d_ops, &e->d_tok_code, &e->d_tok_name, &e->d_tok_region,
                  &e->d_dport_begin, &e->d_dports, &e->d_scan_tiles, &e->d_hist})
    cudaFree(b->p);
  for (HostResult *h : e->free_results) {
    for (DBuf *b : {&h->status_ga, &h->status_r53, &h->derived, &h->ops, &h->tok_code, &h->tok_name, &h->tok_region, &h->dport_begin, &h->dports, &h->obj_gid}) cudaFreeHost(b->p);
    delete h;
  }
  for (auto &ev : e->ev)
    if (ev) cudaEventDestroy(ev);
  for (auto &ev : e->event_pool) cudaEventDestroy(ev);
  if (e->stream) cudaStreamDestroy(e->stream);
  delete e;
}

int gar_snapshot_load(gar_engine *e, const gar_objects *desired, const gar_actual *actual) {
  return guarded(e, [&] {
    do_load(e, desired, actual);
    e->T.cluster = (const u8 *)e->cluster_dev.p;
    e->T.cluster_len = (u32)e->cluster.size();
  });
}

int gar_snapshot_attach_device(gar_engine *e, const gar_objects *desired, const gar_actual *actual) {
  return guarded(e, [&] {
    if (!desired || !actual) throw InvalidError{"NULL table struct"};
    e->graph_drop();
    delete e->pipe;
    e->pipe = nullptr;
    e->T.o = *desired;
    e->T.a = *actual;
    e->T.cluster = (const u8 *)e->cluster_dev.p;
    e->T.cluster_len = (u32)e->cluster.size();
    e->input_bytes = table_bytes(desired, actual);
    e->ms_h2d = 0;
    e->loaded = true;
    e->attached = true;
    e->slice = e->T;
    e->shard_home = false;
    e->shard_round = 0;
  });
}

int gar_diff(gar_engine *e, gar_changeset *out) {
  if (!out) return GAR_E_INVALID;
  return guarded(e, [&] { do_diff(e, out, true); });
}

int gar_diff_device(gar_engine *e, gar_changeset *out) {
  if (!out) return GAR_E_INVALID;
  return guarded(e, [&] { do_diff(e, out, false); });
}

int gar_diff_keys(gar_engine *e, const gar_keyset *keys, gar_changeset *out) {
  if (!out || !keys) return GAR_E_INVALID;
  return guarded(e, [&] { do_diff(e, out, true, keys); });
}

int gar_bindings_diff(gar_engine *e, const gar_bindings *bindings, gar_changeset *out) {
  if (!out || !bindings) return GAR_E_INVALID;
  return guarded(e, [&] { do_diff(e, out, true, nullptr, bindings); });
}

int gar_shard_route(gar_engine *e, const gar_shard *shard, int round, uint64_t *meta, uint64_t *send_bytes) {
  if (!shard || !meta || !send_bytes) return GAR_E_INVALID;
  return guarded(e, [&] {
    if (!e->loaded) throw InvalidError{"no slice loaded"};
    if (shard->n_ranks < 1 || shard->n_ranks > GAR_SHARD_MAX_RANKS || shard->rank >= shard->n_ranks) throw InvalidError{"bad gar_shard"};
    CK(cudaSetDevice(e->device));
    if (!e->sharder) e->sharder = new Sharder<gar_engine>(*e);
    u32 l0 = e->launches;
    if (round == 1) {
      e->marks.clear();
      e->events_used = 0;
      e->stage_depth = 0;
      e->shard_reported = false;
      e->shard_launches = 0;
      e->slice.cluster = (const u8 *)e->cluster_dev.p;
      e->slice.cluster_len = (u32)e->cluster.size();
      e->sharder->route1(e->slice, *shard, meta, send_bytes);
      e->shard_round = 1;
    } else if (round == 2) {
      if (e->shard_round != 2) throw InvalidError{"gar_shard_route(2) needs the round-1 blobs unpacked first"};
      e->sharder->route2(meta, send_bytes);
      e->shard_round = 3;
    } else {
      throw InvalidError{"round must be 1 or 2"};
    }
    e->shard_launches += e->launches - l0;
    CK(cudaStreamSynchronize(e->stream));
  });
}

int gar_shard_pack(gar_engine *e, void *send) {
  return guarded(e, [&] {
    if (e->shard_round != 1 && e->shard_round != 3) throw InvalidError{"gar_shard_pack without a routed plan"};
    CK(cudaSetDevice(e->device));
    u32 l0 = e->launches;
    e->sharder->pack((u8 *)send);
    e->shard_launches += e->launches - l0;
    CK(cudaStreamSynchronize(e->stream));  // the host hands `send` to the exchange next
    CK(cudaGetLastError());
  });
}

int gar_shard_unpack(gar_engine *e, int round, const void *recv, const uint64_t *recv_meta) {
  if (!recv_meta) return GAR_E_INVALID;
  return guarded(e, [&] {
    CK(cudaSetDevice(e->device));
    u32 l0 = e->launches;
    if (round == 1 && e->shard_round == 1) {
      if (e->sharder->unpack1((const u8 *)recv, recv_meta) != GAR_OK) throw InvalidError{e->sharder->contract_error};
      e->shard_round = 2;
    } else if (round == 2 && e->shard_round == 3) {
      if (e->sharder->unpack2((const u8 *)recv, recv_meta) != GAR_OK) throw InvalidError{e->sharder->contract_error};
      delete e->pipe;
      e->pipe = nullptr;
      e->T = e->sharder->H;
      e->shard_home = true;
      e->shard_round = 4;
    } else {
      throw InvalidError{"gar_shard_unpack out of sequence"};
    }
    e->shard_launches += e->launches - l0;
    CK(cudaStreamSynchronize(e->stream));
    CK(cudaGetLastError());
  });
}

uint64_t gar_shard_blob_bytes(const uint64_t *meta_row) { return meta_row ? blob_bytes(meta_row) : 0; }

int gar_shard_arena(gar_engine *e, int round, uint64_t need_bytes, void **arena, uint8_t *handle, uint64_t *capacity) {
  if (!arena || !handle || (round != 1 && round != 2)) return GAR_E_INVALID;
  return guarded(e, [&] {
    CK(cudaSetDevice(e->device));
    DBuf &b = e->peer_arena[round - 1];
    if (b.cap < need_bytes + 64) {
      CK(cudaStreamSynchronize(e->stream));  // nobody may still be reading the old arena (the caller's barrier covers the peers)
      if (b.p) CK(cudaFree(b.p));
      b.p = nullptr;
      b.cap = 0;
      size_t want = (size_t)(need_bytes + need_bytes / 4 + 4096);
      CK(cudaMalloc(&b.p, want));  // plain cudaMalloc: the only kind of allocation CUDA IPC can export
      b.cap = want;
    }
    gar_engine::PeerHandle h{};
    h.magic = 0x6761725F70656572ull;  // "gar_peer"
    h.pid = (u64)getpid();
    h.ptr = (u64)(uintptr_t)b.p;
    h.cap = b.cap;
    CK(cudaIpcGetMemHandle(&h.ipc, b.p));
    memset(handle, 0, GAR_SHARD_HANDLE_BYTES);
    memcpy(handle, &h, sizeof(h));
    *arena = b.p;
    if (capacity) *capacity = b.cap;
  });
}

int gar_shard_open_peers(gar_engine *e, int round, const uint8_t *handles) {
  if (!handles || (round != 1 && round != 2)) return GAR_E_INVALID;
  return guarded(e, [&] {
    if (!e->sharder || e->shard_round == 0) throw InvalidError{"gar_shard_open_peers before gar_shard_route"};
    CK(cudaSetDevice(e->device));
    const u32 G = e->sharder->G, me = e->sharder->cfg.rank;
    const int r = round - 1;
    for (u32 k = 0; k < G; k++) {
      gar_engine::PeerHandle h;
      memcpy(&h, handles + (size_t)k * GAR_SHARD_HANDLE_BYTES, sizeof(h));
      if (h.magic != 0x6761725F70656572ull) throw InvalidError{"bad peer handle"};
      if (k == me || h.pid == (u64)getpid()) {  // this process's own memory (several engines in one process: tests): no IPC needed
        e->peer_ptr[r][k] = (u8 *)(uintptr_t)h.ptr;
        continue;
      }
      if (e->peer_mapped[r][k] && !memcmp(&e->peer_seen[r][k], &h, sizeof(h))) continue;  // still the mapping we have
      if (e->peer_mapped[r][k]) {
        CK(cudaIpcCloseMemHandle(e->peer_ptr[r][k]));
        e->peer_mapped[r][k] = false;
      }
      void *p = nullptr;
      CK(cudaIpcOpenMemHandle(&p, h.ipc, cudaIpcMemLazyEnablePeerAccess));
      e->peer_ptr[r][k] = (u8 *)p;
      e->peer_mapped[r][k] = true;
      e->peer_seen[r][k] = h;
    }
  });
}

int gar_shard_pack_peers(gar_engine *e, int round, const uint64_t *all_meta) {
  if (!all_meta || (round != 1 && round != 2)) return GAR_E_INVALID;
  return guarded(e, [&] {
    if (e->shard_round != 1 && e->shard_round != 3) throw InvalidError{"gar_shard_pack_peers without a routed plan"};
    CK(cudaSetDevice(e->device));
    const u32 G = e->sharder->G, me = e->sharder->cfg.rank;
    const int r = round - 1;
    u8 *bases[GAR_SHARD_MAX_RANKS] = {};
    for (u32 d = 0; d < G; d++) {
      if (!e->peer_ptr[r][d]) throw InvalidError{"gar_shard_pack_peers: a peer arena is not mapped (gar_shard_open_peers)"};
      u64 off = 0;
      for (u32 s = 0; s < me; s++) off += blob_bytes(all_meta + ((size_t)s * G + d) * GAR_SHARD_META_WORDS);
      bases[d] = e->peer_ptr[r][d] + off;
    }
    u32 l0 = e->launches;
    if (G == 1) {
      e->sharder->pack_to(bases);
    } else {
      // own blob: packed in place.  The others: packed into the local stage, then pushed by k_peer_push
      u64 stage_off[GAR_SHARD_MAX_RANKS + 1] = {0};
      for (u32 d = 0; d < G; d++)
        stage_off[d + 1] = stage_off[d] + (d == me ? 0 : blob_bytes(all_meta + ((size_t)me * G + d) * GAR_SHARD_META_WORDS));
      DBuf &st = e->peer_stage;
      if (st.cap < stage_off[G] + 64) {
        CK(cudaStreamSynchronize(e->stream));
        if (st.p) CK(cudaFree(st.p));
        st.p = nullptr;
        st.cap = 0;
        size_t want = (size_t)(stage_off[G] + stage_off[G] / 4 + 4096);
        CK(cudaMalloc(&st.p, want));
        st.cap = want;
      }
      u8 *peer_base[GAR_SHARD_MAX_RANKS] = {};
      for (u32 d = 0; d < G; d++) {
        peer_base[d] = bases[d];
        if (d != me) bases[d] = (u8 *)st.p + stage_off[d];
      }
      if (!e->peer_push_stream) {
        int lo = 0, hi = 0;
        CK(cudaDeviceGetStreamPriorityRange(&lo, &hi));
        CK(cudaStreamCreateWithPriority(&e->peer_push_stream, cudaStreamNonBlocking, hi));
      }
      u64 sent[GAR_SHARD_MAX_RANKS] = {0};
      size_t ev_used = 0;
      const u64 kGroupBytes = 48ull << 20;  // start a transfer once this much (over all destinations) is packed
      e->sharder->pack_to(bases, [&](int lvl, const u64 *end) {
        u64 pending = 0;
        for (u32 d = 0; d < G; d++)
          if (d != me) pending += end[d] - sent[d];
        if (!pending || (lvl < (int)L_NLEVELS && pending < kGroupBytes)) return;
        if (ev_used == e->peer_ev.size()) {
          cudaEvent_t ev;
          CK(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
          e->peer_ev.push_back(ev);
        }
        cudaEvent_t ev = e->peer_ev[ev_used++];
        CK(cudaEventRecord(ev, e->stream));
        PushDesc pd{};
        u32 cnt = 0;
        for (u32 k = 1; k < G; k++) {  // rank r starts with r+1: no destination is everybody's first
          u32 d = (me + k) % G;
          if (end[d] == sent[d]) continue;
          pd.src[cnt] = (const uint4 *)(bases[d] + sent[d]);
          pd.dst[cnt] = (uint4 *)(peer_base[d] + sent[d]);
          pd.n16[cnt] = (end[d] - sent[d]) >> 4;  // blob sections are multiples of 16 bytes (sh_align)
          sent[d] = end[d];
          cnt++;
        }
        CK(cudaStreamWaitEvent(e->peer_push_stream, ev, 0));
        k_peer_push<<<dim3(PUSH_BLOCKS, cnt), PUSH_THREADS, 0, e->peer_push_stream>>>(pd);
        e->launches++;
      });
      CK(cudaStreamSynchronize(e->peer_push_stream));
    }
    e->shard_launches += e->launches - l0;
    CK(cudaStreamSynchronize(e->stream));  // the stores are performed: after the ranks' barrier every arena is complete
    CK(cudaGetLastError());
  });
}

void gar_changeset_free(gar_engine *e, gar_changeset *cs) {
  if (!e || !cs) return;
  std::lock_guard<std::mutex> lk(e->mu);
  if (cs->opaque) e->free_results.push_back((HostResult *)cs->opaque);
  memset(cs, 0, sizeof(*cs));
}

const char *gar_last_error(const gar_engine *e) { return e ? e->err.c_str() : g_create_error.c_str(); }

const char *gar_version(void) { return GAR_VERSION_STRING; }

uint64_t gar_algorithmic_bytes(const gar_engine *e, const gar_changeset *cs) {
  if (!e || !cs) return 0;
  return e->input_bytes + 2ull * 4 * cs->n_objects + sizeof(gar_op) * cs->n_ops;
}

uint32_t gar_last_stage_timings(gar_engine *e, gar_stage_timing *out, uint32_t cap) {
  if (!e) return 0;
  std::lock_guard<std::mutex> lk(e->mu);
  uint32_t n = (uint32_t)e->last_timings.size();
  for (uint32_t i = 0; i < n && i < cap; i++) out[i] = e->last_timings[i];
  return n;
}

uint32_t gar_last_counters(gar_engine *e, uint64_t *out, uint32_t cap) {
  if (!e || !out) return 0;
  std::lock_guard<std::mutex> lk(e->mu);
  uint32_t n = cap < GAR_CTR_N ? cap : (uint32_t)GAR_CTR_N;
  for (uint32_t i = 0; i < n; i++) out[i] = e->last_counters[i];
  return n;
}

}  // extern "C"
