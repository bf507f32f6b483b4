// peer.cu — the GPUs of one box working on ONE dist call (SURVEY.md §8e: ref rows sharded, query HVs
// broadcast, hit lists gathered).  The reference has nothing to replace here: dist is a single rayon
// loop over all pairs on the host (src/dist.rs:231-294).
//
// Every member GPU owns a "window" of device memory that all other members can address over NVLink
// (one process per GPU: cudaIpc handles; one process driving several GPUs: peer access).  A sharded
// dist then needs no collective library on its data path, and the exchange overlaps the compute:
//   1. each member turns ITS rows into the operand form of the tensor kernel (one s8 plane + per-row
//      constants, or two s8 limb planes) inside its own window and PUSHES them, in up to 4 chunks of
//      about 2 MB or more, with plain 16-byte stores over NVLink to the same offsets of other windows:
//      1 byte per element instead of the 2 of the int16 rows, no pre-pass replicated on every GPU.
//      The last pusher warp through with a chunk raises that chunk's ARRIVAL FLAG in the destination
//      windows (fence + st.release.sys, one lane per window);
//   2. every member launches the dist kernel at once.  Its tiles come from a host-built list.
//      All-vs-all with row blocks that are multiples of 256 rows ("ring"): the
//      block pair (a, b) is computed by the member from which the other block is at most N/2 steps
//      AHEAD on the ring (the pair exactly N/2 apart is split tile by tile), so a member's rows go to
//      floor(N/2) members instead of N - 1 - half the NVLink bytes.  Otherwise the
//      non-empty tiles are dealt round-robin (tile t to member t mod N) and every chunk goes to
//      everybody.  A member's tiles are ordered own rows, chunk 0 of everybody, chunk 1 ...  The kernel's TMA
//      producer waits for the arrival flags a tile needs (ld.acquire.sys on its own window, bounded) -
//      tiles are computed while later chunks are still crossing NVLink.  ref x query: the member's own
//      (resident) ref rows against all queries, same mechanism on the query side;
//   3. hits are appended straight into the ROOT's hit list - its window, or a host buffer every member
//      has mapped - with one atomic on the root's counter per evaluated candidate list;
//   4. one flag barrier at the end (st.release.sys / ld.acquire.sys, bounded spin); the root's stream
//      then owns the complete hit list.
// Measured on 2 B200s (tools/ipc_probe.cu): push of a 21 MB slice + two barriers 49 us (NCCL all_gather
// of the same plane 69 us), flag barrier 6.3 us.
#include <algorithm>
#include <cmath>
#include <cstring>
#include <functional>
#include <string>
#include <thread>
#include <vector>

#include "hg_common.cuh"

namespace {

constexpr size_t OFF_FLAGS = 0;      // u32[HG_MAX_PEERS]: flags[r] = last barrier epoch member r has reached
constexpr size_t OFF_SEQ = 32;       // u32[2]: [0] sharded dist launches so far (what the arrival flags count), [1] barriers so far
constexpr size_t OFF_STATUS = 64;    // u32: a barrier / an arrival wait of this member timed out
constexpr size_t OFF_COUNT = 128;    // u64: hits in THIS member's list
constexpr size_t OFF_TOTAL = 136;    // u64: hits of all members gathered so far (the root's is the one in use)
constexpr size_t OFF_STATS_Q = 256;  // u32[HG_MAX_PEERS][4]: pre-pass statistics of the gathered (query) matrix, one set per member
constexpr size_t OFF_STATS_R = 384;  // u32[HG_MAX_PEERS][4]: ... of the members' own ref rows (ref x query)
constexpr size_t OFF_READY = 512;    // u32[32]: arrival flags, flag m * 4 + c = sequence number of the last call for which chunk c of member m's rows is here
constexpr size_t OFF_DONE = 640;     // u32[HG_PUSH_UNITS]: pusher warps / CTAs through with push unit u (local use)
constexpr size_t OFF_DBG = 768;      // u64[32]: timeline stamps of the last sharded dist (globaltimer ns; HG_PEER_TIMELINE=1)
constexpr size_t OFF_START = 1024;   // u32[HG_MAX_PEERS]: start flags, flag m = sequence number of the last call whose start set of member m is here
constexpr int N_CHUNKS = HG_PUSH_CHUNKS;
constexpr uint64_t CHUNK_TARGET_BYTES = 2u << 20;  // a member's block is cut into chunks of at least about this much
static_assert(OFF_DONE + 4 * HG_PUSH_UNITS <= OFF_DBG, "header layout");
constexpr size_t OFF_HITS = 4096;    // hg_hit[cap]

struct PeerPtrs { uint8_t *p[HG_MAX_PEERS]; };

__device__ __forceinline__ unsigned long long global_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}

// One warp: lane t tells member t that this member has reached `epoch`, then waits until member t has.
// Everything this stream wrote before (its pushes) is complete when the kernel starts; the fence + release
// order it before the flag.  The spin is bounded: a member that never arrives (a failed launch, a dead
// process) turns into an error status instead of a hung GPU.
__global__ void peer_barrier_kernel(PeerPtrs w, int rank, int world, unsigned long long timeout_ns, unsigned long long *dbg) {
  const int t = threadIdx.x;
  if (dbg && t == 0) dbg[13] = global_ns();
  uint32_t *ep = reinterpret_cast<uint32_t *>(w.p[rank] + OFF_SEQ) + 1;  // barriers so far: device-resident, so that the
  uint32_t epoch = 0;                                                    // launch sequence can be replayed as a CUDA graph
  if (t == 0) { epoch = *ep + 1; *ep = epoch; }
  epoch = __shfl_sync(0xffffffffu, epoch, 0);
  if (t >= world) return;
  __threadfence_system();
  uint32_t *theirs = reinterpret_cast<uint32_t *>(w.p[t] + OFF_FLAGS) + rank;
  asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(theirs), "r"(epoch) : "memory");
  const uint32_t *mine = reinterpret_cast<const uint32_t *>(w.p[rank] + OFF_FLAGS) + t;
  const unsigned long long t0 = global_ns();
  for (;;) {
    uint32_t v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(mine) : "memory");
    if ((int32_t)(v - epoch) >= 0) break;
    if (global_ns() - t0 > timeout_ns) {
      atomicExch(reinterpret_cast<uint32_t *>(w.p[rank] + OFF_STATUS), 1u);
      break;
    }
  }
  if (dbg) atomicMax(dbg + 14, global_ns());  // when the last member was seen
}

// First node of a sharded dist on every member: next sequence number, my hit counter and my pre-pass statistics reset
// (the cursor of my outlier entries starts at my share of the entry space), the root's gather counter reset.
__global__ void peer_tick_kernel(uint8_t *W, int rank, int is_root, uint32_t entry_base, int timeline) {
  if (timeline) {  // stamps 0..15 of this call; [16] keeps the previous call's barrier exit (the members' common time base)
    unsigned long long *dbg = reinterpret_cast<unsigned long long *>(W + OFF_DBG);
    if (threadIdx.x == 0) dbg[16] = dbg[14];
    __syncwarp();
    if (threadIdx.x < 16) dbg[threadIdx.x] = threadIdx.x == 0 ? global_ns() : 0ull;
  }
  if (threadIdx.x == 0) {
    uint32_t *seq = reinterpret_cast<uint32_t *>(W + OFF_SEQ);
    *seq = *seq + 1;
    *reinterpret_cast<unsigned long long *>(W + OFF_COUNT) = 0ull;
    if (is_root) *reinterpret_cast<unsigned long long *>(W + OFF_TOTAL) = 0ull;
  }
  if (threadIdx.x < 4) {
    reinterpret_cast<uint32_t *>(W + OFF_STATS_Q)[4 * rank + threadIdx.x] = threadIdx.x == 2 ? entry_base : 0u;
    reinterpret_cast<uint32_t *>(W + OFF_STATS_R)[4 * rank + threadIdx.x] = 0u;
  }
}

// After a member's dist kernel: its hit list (in its own window - local atomics, local stores while the tiles were
// computed) moves to the root in ONE piece: one atomic on the root's counter reserves the room, then coalesced 16-byte
// stores - over NVLink into the root's gather list, or over this GPU's own PCIe link into a host buffer that every
// member has mapped.
__global__ void peer_flush_kernel(uint8_t *W, unsigned long long *root_total, hg_hit *dst, unsigned long long cap, int timeline) {
  __shared__ unsigned long long s_base;
  if (timeline && blockIdx.x == 0 && threadIdx.x == 0) reinterpret_cast<unsigned long long *>(W + OFF_DBG)[12] = global_ns();
  const unsigned long long cnt = *reinterpret_cast<const unsigned long long *>(W + OFF_COUNT);
  const unsigned long long n = cnt < cap ? cnt : cap;  // records beyond my list's capacity were counted, not stored
  // every block moves a contiguous slice of my list and reserves exactly that much room on the root
  const unsigned long long per = (n + gridDim.x - 1) / gridDim.x;
  const unsigned long long lo = per * blockIdx.x < n ? per * blockIdx.x : n, hi = lo + per < n ? lo + per : n;
  const unsigned long long extra = blockIdx.x == 0 ? cnt - n : 0;  // overflow of my own list still counts towards the need
  if (hi == lo && extra == 0) return;
  if (threadIdx.x == 0) s_base = atomicAdd(root_total, hi - lo + extra);
  __syncthreads();
  const unsigned long long base = s_base;
  const uint4 *src = reinterpret_cast<const uint4 *>(W + OFF_HITS);
  uint4 *out = reinterpret_cast<uint4 *>(dst);
  for (unsigned long long i = lo + threadIdx.x; i < hi; i += blockDim.x)
    if (base + (i - lo) < cap) out[base + (i - lo)] = src[i];
}

// Copies byte ranges of this member's window to the same offsets of the windows in `dest`.
struct PushRange { uint64_t off, bytes; };  // 4-byte granular; ranges that are 16-byte aligned go as uint4
struct PushArgs { PushRange r[HG_PUSH_RANGES]; int n; };

__global__ void __launch_bounds__(256) peer_push_kernel(PeerPtrs w, int rank, int world, PushArgs a, uint32_t dest, uint64_t flag_off, uint32_t *done) {
  const uint32_t seq = *reinterpret_cast<const uint32_t *>(w.p[rank] + OFF_SEQ);
  const size_t tid = (size_t)blockIdx.x * blockDim.x + threadIdx.x, nth = (size_t)gridDim.x * blockDim.x;
  for (int k = 0; k < a.n; ++k) {
    const uint64_t off = a.r[k].off, bytes = a.r[k].bytes;
    if (((off | bytes) & 15) == 0) {
      const uint4 *src = reinterpret_cast<const uint4 *>(w.p[rank] + off);
      const size_t n16 = bytes / 16;
      for (size_t i = tid; i < n16; i += 4 * nth) {  // four loads in flight per thread, then their stores to every peer
        uint4 v[4];
#pragma unroll
        for (int u = 0; u < 4; ++u)
          if (i + u * nth < n16) v[u] = src[i + u * nth];
#pragma unroll
        for (int u = 0; u < 4; ++u)
          if (i + u * nth < n16)
            for (int m = 0; m < world; ++m)
              if (dest >> m & 1u) reinterpret_cast<uint4 *>(w.p[m] + off)[i + u * nth] = v[u];
      }
    } else {
      const uint32_t *src = reinterpret_cast<const uint32_t *>(w.p[rank] + off);
      for (size_t i = tid; i < bytes / 4; i += nth) {
        const uint32_t v = src[i];
        for (int m = 0; m < world; ++m)
          if (dest >> m & 1u) reinterpret_cast<uint32_t *>(w.p[m] + off)[i] = v;
      }
    }
  }
  // the last CTA to finish raises the unit's flag in the destination windows (one thread per window: the release
  // stores are in flight together)
  __shared__ uint32_t s_last;
  __threadfence_system();
  __syncthreads();
  if (threadIdx.x == 0) {
    const uint32_t prev = atomicAdd(done, 1u);
    s_last = prev == gridDim.x - 1;
    if (s_last) *done = 0;
  }
  __syncthreads();
  if (s_last && (int)threadIdx.x < world && (dest >> threadIdx.x & 1u)) {
    __threadfence_system();
    uint32_t *f = reinterpret_cast<uint32_t *>(w.p[threadIdx.x] + flag_off);
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(f), "r"(seq) : "memory");
  }
}

inline uint64_t align_up(uint64_t x, uint64_t a) { return (x + a - 1) / a * a; }

// where the pieces of one sharded dist live inside every window (same call arguments -> same layout everywhere)
struct ShardLayout {
  uint64_t gather, norm, arrays, entries, plane, end;
  uint32_t set_cap;
};
// [header | my hit list | gathered hit list (root; absent when the hits go to a mapped host buffer) | norms | operands]
ShardLayout make_layout(int world, uint32_t n_total, uint32_t hv_d, uint64_t cap, int n_planes, bool mapped) {
  ShardLayout l;
  l.gather = align_up(OFF_HITS + cap * sizeof(hg_hit), 1024);
  l.norm = align_up(l.gather + (mapped ? 0 : cap * sizeof(hg_hit)), 1024);
  l.arrays = align_up(l.norm + (uint64_t)n_total * 4, 256);
  l.set_cap = n_planes == 1 ? hg_narrow_set_cap(n_total) : 0;
  l.entries = align_up(l.arrays + (n_planes == 1 ? hg_narrow_arrays_bytes(n_total) : 0), 256);
  l.plane = align_up(l.entries + (uint64_t)world * l.set_cap * 4, 1024);
  l.end = l.plane + (n_planes == 1 ? (uint64_t)n_total * hv_d : hg_tc_mat_bytes(n_total, hv_d)) + 1024;  // two limb planes: + row sums
  return l;
}

}  // namespace

struct TileKey {  // what a cached tile list was built for
  int sym, path;
  uint32_t n_ref, n_qry, tr, tc, hv_d;
  uint32_t qb[HG_MAX_PEERS + 1];
};

struct hg_peer {
  hg_ctx *ctx = nullptr;
  int rank = 0, world = 1;
  int local = 0;                 // members driven by one process (peer access) rather than one process per GPU (cudaIpc)
  uint64_t window_bytes = 0;
  uint8_t *win[HG_MAX_PEERS] = {};  // every member's window as THIS member addresses it (win[rank] = its own allocation)
  bool opened[HG_MAX_PEERS] = {};
  bool connected = false;
  unsigned long long timeout_ns = 0;
  int last_ring = 0;  // the last sharded dist used the ring ownership
  int timeline = 0;  // HG_PEER_TIMELINE=1: the kernels of a sharded dist stamp globaltimer values into the window (hg_peer_timeline)
  uint8_t *h_hdr = nullptr;  // pinned copy of window bytes [OFF_STATUS, OFF_STATUS + 128): status word and hit counters of the
                             // last call, written by the call's last node
  // The launch sequence of a sharded dist with asserted path (same pointers, same shapes, call after call) is captured
  // once and replayed as a CUDA graph: one launch instead of ~10, no gaps between the nodes.
  cudaGraphExec_t graph = nullptr;
  std::vector<uint8_t> graph_key, last_key;
  unsigned graph_nodes = 0;
  // the last sharded dist
  int root = 0;
  uint64_t cap = 0;
  hg_hit *mapped_hits = nullptr;  // hits went to a host buffer every member has mapped, not to the root's window
  uint64_t gather_off = 0;        // where the root's gathered list starts in its window
  // this member's tile list (host copy + what it was built for; the device copy lives in scratch slot HG_S_TILES)
  std::vector<uint2> tiles;
  TileKey tiles_key = {};
  bool tiles_valid = false, tiles_on_device = false;
  // stage boundaries of the last sharded dist (recorded when the context profiles): start | operands ready | pushed |
  // kernel done | final barrier passed
  cudaEvent_t ev[6] = {};
  int ev_n = 0;
};
#define PEER_PROF(p, i)                                                      \
  do {                                                                       \
    if ((p)->ctx->prof) {                                                    \
      if (!(p)->ev[i]) cudaEventCreate(&(p)->ev[i]);                         \
      cudaEventRecord((p)->ev[i], (p)->ctx->stream);                         \
      (p)->ev_n = (i) + 1;                                                   \
    }                                                                        \
  } while (0)

static PeerPtrs peer_ptrs(const hg_peer *p) {
  PeerPtrs w;
  for (int r = 0; r < HG_MAX_PEERS; ++r) w.p[r] = r < p->world ? p->win[r] : nullptr;
  return w;
}

extern "C" uint64_t hg_peer_window_need(uint32_t gathered_rows, uint32_t hv_d, uint64_t hit_cap) {
  const ShardLayout a = make_layout(HG_MAX_PEERS, gathered_rows, hv_d, hit_cap, 1, false), b = make_layout(HG_MAX_PEERS, gathered_rows, hv_d, hit_cap, 2, false);
  return std::max(a.end, b.end) + 4096;
}

static int peer_alloc(hg_ctx *ctx, int rank, int world, uint64_t window_bytes, hg_peer **out) {
  if (!ctx || !out) { hg_set_error("hg_peer_create: NULL argument"); return HG_E_INVALID; }
  if (world < 1 || world > HG_MAX_PEERS || rank < 0 || rank >= world) { hg_set_error("hg_peer_create: rank %d of %d (at most %d members)", rank, world, HG_MAX_PEERS); return HG_E_INVALID; }
  if (window_bytes < OFF_HITS + 4096) window_bytes = OFF_HITS + 4096;
  HG_CUDA(cudaSetDevice(ctx->device));
  hg_peer *p = new hg_peer();
  p->ctx = ctx;
  p->rank = rank;
  p->world = world;
  p->window_bytes = window_bytes;
  p->timeout_ns = 10ull * 1000000000ull;
  if (const char *e = getenv("HG_PEER_TIMEOUT_MS")) p->timeout_ns = (unsigned long long)std::max(1, atoi(e)) * 1000000ull;
  if (const char *e = getenv("HG_PEER_TIMELINE")) p->timeline = atoi(e) != 0;
  void *w = nullptr;
  cudaError_t e = cudaMalloc(&w, window_bytes);
  if (e != cudaSuccess) { delete p; return hg_cuda_fail(e, "cudaMalloc(window)", __FILE__, __LINE__); }
  e = cudaMemset(w, 0, OFF_HITS);
  if (e == cudaSuccess) e = cudaDeviceSynchronize();
  if (e != cudaSuccess) { cudaFree(w); delete p; return hg_cuda_fail(e, "cudaMemset(window)", __FILE__, __LINE__); }
  p->win[rank] = (uint8_t *)w;
  e = cudaMallocHost(&p->h_hdr, 128);
  if (e != cudaSuccess) { cudaFree(w); delete p; return hg_cuda_fail(e, "cudaMallocHost", __FILE__, __LINE__); }
  memset(p->h_hdr, 0, 128);
  *out = p;
  return HG_OK;
}

// One process per GPU: allocate this member's window and return the handle the other members open.
extern "C" int hg_peer_create(hg_ctx *ctx, int rank, int world, uint64_t window_bytes, uint8_t handle_out[HG_IPC_HANDLE_BYTES],
                              hg_peer **out) {
  static_assert(sizeof(cudaIpcMemHandle_t) == HG_IPC_HANDLE_BYTES, "IPC handle size");
  if (!handle_out) { hg_set_error("hg_peer_create: handle_out is NULL"); return HG_E_INVALID; }
  int rc = peer_alloc(ctx, rank, world, window_bytes, out);
  if (rc) return rc;
  cudaIpcMemHandle_t h;
  cudaError_t e = cudaIpcGetMemHandle(&h, (*out)->win[rank]);
  if (e != cudaSuccess) { hg_peer_destroy(*out); *out = nullptr; return hg_cuda_fail(e, "cudaIpcGetMemHandle", __FILE__, __LINE__); }
  memcpy(handle_out, &h, HG_IPC_HANDLE_BYTES);
  if (world == 1) (*out)->connected = true;
  return HG_OK;
}

// `handles`: world x HG_IPC_HANDLE_BYTES in rank order (this member's own entry is ignored).  Every member must have
// created its window before anyone connects (the caller's bootstrap - an all-gather of the handles - implies that).
extern "C" int hg_peer_connect(hg_peer *p, const uint8_t *handles) {
  if (!p || !handles) { hg_set_error("hg_peer_connect: NULL argument"); return HG_E_INVALID; }
  if (p->local) { hg_set_error("hg_peer_connect: a single-process group is connected at creation"); return HG_E_INVALID; }
  HG_CUDA(cudaSetDevice(p->ctx->device));
  for (int r = 0; r < p->world; ++r) {
    if (r == p->rank || p->opened[r]) continue;
    cudaIpcMemHandle_t h;
    memcpy(&h, handles + (size_t)r * HG_IPC_HANDLE_BYTES, HG_IPC_HANDLE_BYTES);
    void *w = nullptr;
    HG_CUDA(cudaIpcOpenMemHandle(&w, h, cudaIpcMemLazyEnablePeerAccess));
    p->win[r] = (uint8_t *)w;
    p->opened[r] = true;
  }
  p->connected = true;
  return HG_OK;
}

// One process driving `world` GPUs: windows with mutual peer access.  out[0..world) receives the members.
extern "C" int hg_peer_create_local(hg_ctx *const *ctxs, int world, uint64_t window_bytes, hg_peer **out) {
  if (!ctxs || !out) { hg_set_error("hg_peer_create_local: NULL argument"); return HG_E_INVALID; }
  if (world < 1 || world > HG_MAX_PEERS) { hg_set_error("hg_peer_create_local: %d members (at most %d)", world, HG_MAX_PEERS); return HG_E_INVALID; }
  for (int r = 0; r < world; ++r) out[r] = nullptr;
  int rc = HG_OK;
  for (int r = 0; r < world && !rc; ++r) rc = peer_alloc(ctxs[r], r, world, window_bytes, &out[r]);
  for (int r = 0; r < world && !rc; ++r) {
    cudaSetDevice(ctxs[r]->device);
    for (int m = 0; m < world && !rc; ++m) {
      if (m == r || ctxs[m]->device == ctxs[r]->device) continue;
      int can = 0;
      cudaDeviceCanAccessPeer(&can, ctxs[r]->device, ctxs[m]->device);
      if (!can) { hg_set_error("device %d cannot address device %d (no peer access)", ctxs[r]->device, ctxs[m]->device); rc = HG_E_UNSUPPORTED; break; }
      const cudaError_t e = cudaDeviceEnablePeerAccess(ctxs[m]->device, 0);
      if (e == cudaErrorPeerAccessAlreadyEnabled) cudaGetLastError();
      else if (e != cudaSuccess) rc = hg_cuda_fail(e, "cudaDeviceEnablePeerAccess", __FILE__, __LINE__);
    }
  }
  if (rc) {
    for (int r = 0; r < world; ++r) if (out[r]) { hg_peer_destroy(out[r]); out[r] = nullptr; }
    return rc;
  }
  for (int r = 0; r < world; ++r) {
    out[r]->local = 1;
    out[r]->connected = true;
    for (int m = 0; m < world; ++m) out[r]->win[m] = out[m]->win[m];
  }
  return HG_OK;
}

extern "C" void hg_peer_destroy(hg_peer *p) {
  if (!p) return;
  cudaSetDevice(p->ctx->device);
  cudaStreamSynchronize(p->ctx->stream);
  for (int r = 0; r < p->world; ++r)
    if (p->opened[r]) cudaIpcCloseMemHandle(p->win[r]);
  if (p->win[p->rank]) cudaFree(p->win[p->rank]);
  for (int i = 0; i < 6; ++i) if (p->ev[i]) cudaEventDestroy(p->ev[i]);
  if (p->graph) cudaGraphExecDestroy(p->graph);
  if (p->h_hdr) cudaFreeHost(p->h_hdr);
  delete p;
}

extern "C" int hg_peer_rank(const hg_peer *p) { return p ? p->rank : -1; }
extern "C" int hg_peer_world(const hg_peer *p) { return p ? p->world : 0; }

static int peer_barrier(hg_peer *p) {
  peer_barrier_kernel<<<1, 32, 0, p->ctx->stream>>>(peer_ptrs(p), p->rank, p->world, p->timeout_ns,
                                                    p->timeline ? reinterpret_cast<unsigned long long *>(p->win[p->rank] + OFF_DBG) : nullptr);
  p->ctx->launches++;
  HG_CUDA(cudaGetLastError());
  return HG_OK;
}

extern "C" int hg_peer_barrier(hg_peer *p) {
  if (!p || !p->connected) { hg_set_error("hg_peer_barrier: not connected"); return HG_E_INVALID; }
  HG_CUDA(cudaSetDevice(p->ctx->device));
  return peer_barrier(p);
}

// Stand-alone push of one unit (a member that has rows to contribute but no tile to compute - otherwise the dist
// kernel's pusher warps do this, see hg_push_plan): the ranges to the members in `dest`, then the flag at byte offset
// `flag_off` of those windows
static int peer_push(hg_peer *p, const PushArgs &a, uint32_t dest, uint64_t flag_off, int unit) {
  if (p->world == 1) return HG_OK;
  uint64_t bytes = 0;
  for (int k = 0; k < a.n; ++k) bytes += a.r[k].bytes;
  const unsigned blocks = (unsigned)std::min<uint64_t>(std::max<uint64_t>(bytes / (16 * 256 * 4), 1), (uint64_t)p->ctx->sm_count * 4u);
  uint32_t *done = reinterpret_cast<uint32_t *>(p->win[p->rank] + OFF_DONE) + unit;
  peer_push_kernel<<<blocks, 256, 0, p->ctx->stream>>>(peer_ptrs(p), p->rank, p->world, a, dest, flag_off, done);
  p->ctx->launches++;
  HG_CUDA(cudaGetLastError());
  return HG_OK;
}

// ---------------------------------------------------------------------------------------------------
// sharded dist
// ---------------------------------------------------------------------------------------------------
namespace {
struct ShardCall {
  const int16_t *d_ref_hv; const int32_t *d_ref_norm; uint32_t n_ref_local, ref_row0;
  const int16_t *d_qry_hv; const int32_t *d_qry_norm;
  uint32_t qb[HG_MAX_PEERS + 1];  // rows [qb[m], qb[m + 1]) of the gathered (query) matrix are member m's
  uint32_t hv_d, ksize; float ani_th; int symmetric, root; uint64_t cap;
  hg_hit *mapped_hits;
  uint32_t n_qry_total(int world) const { return qb[world]; }
};

// How the members' blocks of the gathered matrix are cut into chunks and who receives them: a pure function of the
// call's shape, so every member derives the same plan.
struct XPlan {
  int world, sym, ring, path;
  uint32_t hv_d;
  int n_chunks[HG_MAX_PEERS];
  uint32_t qb[HG_MAX_PEERS + 1];
};
XPlan make_xplan(int world, int symmetric, int path, uint32_t hv_d, const uint32_t *qb) {
  XPlan x = {};
  x.world = world; x.sym = symmetric; x.path = path; x.hv_d = hv_d;
  bool aligned = true, nonempty = true;
  for (int m = 0; m <= world; ++m) x.qb[m] = qb[m];
  for (int m = 0; m < world; ++m) {
    const uint64_t rows = qb[m + 1] - qb[m], bytes = rows * hv_d * (path == HG_PATH_NARROW ? 1 : 2);
    x.n_chunks[m] = (int)std::min<uint64_t>(std::max<uint64_t>((bytes + CHUNK_TARGET_BYTES - 1) / CHUNK_TARGET_BYTES, 1), N_CHUNKS);
    if (rows == 0) nonempty = false;
    if (m > 0 && qb[m] % 256 != 0) aligned = false;  // a tile (256 rows x 128 or 256 columns) lies inside one block on either side
  }
  x.ring = symmetric && world >= 2 && aligned && nonempty;
  return x;
}
// chunk c of member m's block: rows [chunk_lo(c), chunk_lo(c + 1))
inline uint32_t chunk_lo(const XPlan &x, int m, int c) {
  if (c >= x.n_chunks[m]) return x.qb[m + 1];
  return x.qb[m] + (uint32_t)(((uint64_t)(x.qb[m + 1] - x.qb[m]) * c / x.n_chunks[m]) & ~3ull);
}
// the members that receive member s's rows
inline uint32_t dest_mask(const XPlan &x, int s) {
  uint32_t d = 0;
  if (x.ring) for (int k = 1; k <= x.world / 2; ++k) d |= 1u << ((s - k + x.world) % x.world);
  else for (int m = 0; m < x.world; ++m) if (m != s) d |= 1u << m;
  return d;
}
inline int block_of(const XPlan &x, uint64_t row) {
  int m = 0;
  while (m + 1 < x.world && row >= x.qb[m + 1]) ++m;
  return m;
}
// ring: who computes a tile whose rows lie in block bi and whose columns lie in block bj >= bi
inline int ring_owner(const XPlan &x, int bi, int bj, uint32_t R, uint32_t C) {
  const int d = bj - bi;
  if (2 * d < x.world) return bi;         // bj is d <= N/2 steps ahead of bi
  if (2 * d > x.world) return bj;         // bi is N - d < N/2 steps ahead of bj
  return ((R + C) & 1u) ? bi : bj;        // exactly opposite: both hold the other's block, the tiles alternate
}
// position of (member m, chunk c) in the order in which chunks arrive at member r
inline uint32_t arrival_pos(const XPlan &x, int r, int m, int c) {
  (void)x; (void)r; (void)m;
  return (uint32_t)c;  // every member sends chunk 0 to all its destinations first, then chunk 1, ...
}

// arrival flags (other members' chunks) that rows [x0, x1) of the gathered matrix depend on
uint32_t need_mask(const XPlan &x, int rank, uint64_t x0, uint64_t x1) {
  uint32_t m_ = 0;
  for (int m = 0; m < x.world; ++m) {
    if (m == rank || x.qb[m + 1] <= x0 || x.qb[m] >= x1) continue;
    for (int c = 0; c < x.n_chunks[m]; ++c) {
      const uint64_t lo = chunk_lo(x, m, c), hi = chunk_lo(x, m, c + 1);
      if (lo < hi && lo < x1 && hi > x0) m_ |= 1u << (m * N_CHUNKS + c);
    }
  }
  return m_;
}
}  // namespace

static int shard_check(hg_peer *p, const ShardCall &a) {
  if (!p || !p->connected) { hg_set_error("hg_dist_sharded: the group is not connected"); return HG_E_INVALID; }
  if (a.hv_d == 0 || a.hv_d % 256 != 0) { hg_set_error("hg_dist_sharded: hv_d %u must be a multiple of 256", a.hv_d); return HG_E_INVALID; }
  if (a.root < 0 || a.root >= p->world) { hg_set_error("hg_dist_sharded: root %d of %d", a.root, p->world); return HG_E_INVALID; }
  if (a.qb[0] != 0) { hg_set_error("hg_dist_sharded: qry_bounds[0] must be 0"); return HG_E_INVALID; }
  for (int m = 0; m < p->world; ++m)
    if (a.qb[m + 1] < a.qb[m]) { hg_set_error("hg_dist_sharded: qry_bounds not monotone at member %d", m); return HG_E_INVALID; }
  const uint32_t nl = a.qb[p->rank + 1] - a.qb[p->rank];
  if ((nl && (!a.d_qry_hv || !a.d_qry_norm)) || (!a.symmetric && a.n_ref_local && (!a.d_ref_hv || !a.d_ref_norm))) {
    hg_set_error("hg_dist_sharded: NULL argument"); return HG_E_INVALID;
  }
  if (((uintptr_t)a.d_qry_hv | (uintptr_t)a.d_ref_hv) & 15) { hg_set_error("hg_dist_sharded: HV rows must be 16-byte aligned"); return HG_E_INVALID; }
  if (a.qb[p->world] > 65535u * 128u) { hg_set_error("hg_dist_sharded: more than %u gathered rows", 65535u * 128u); return HG_E_UNSUPPORTED; }
  const bool mp = a.mapped_hits != nullptr;
  const uint64_t need = std::max(make_layout(p->world, a.qb[p->world], a.hv_d, a.cap, 1, mp).end, make_layout(p->world, a.qb[p->world], a.hv_d, a.cap, 2, mp).end);
  if (need > p->window_bytes) {
    hg_set_error("hg_dist_sharded: the windows hold %llu bytes, this call needs %llu (hg_peer_window_need)", (unsigned long long)p->window_bytes,
                 (unsigned long long)need);
    return HG_E_CAPACITY;
  }
  return HG_OK;
}

// Member `rank`'s tiles for a key (pure host logic): its share of the non-empty tiles of the all-vs-all (see the file
// header: ring ownership, or dealt round-robin; ref x query: every tile of the member's own ref rows), each with the
// mask of arrival flags it reads, ordered by when those arrive.
static void plan_tiles(const TileKey &k, int world, int rank, std::vector<uint2> &out) {
  const XPlan x = make_xplan(world, k.sym, k.path, k.hv_d, k.qb);
  const uint32_t gx = (k.n_qry + k.tc - 1) / k.tc, gy = (k.n_ref + k.tr - 1) / k.tr;
  struct T { uint2 e; uint32_t key; };
  std::vector<T> v;
  uint64_t t = 0;
  for (uint32_t R = 0; R < gy; ++R) {
    // symmetric (i0 = j0 = 0): tiles whose largest j is not above their smallest i are empty (as the kernels' cmin)
    uint32_t c0 = 0;
    if (k.sym) c0 = (uint32_t)std::min<uint64_t>(((uint64_t)k.tr * R + 1) / k.tc, gx);
    for (uint32_t C = c0; C < gx; ++C, ++t) {
      if (k.sym) {
        const int owner = x.ring ? ring_owner(x, block_of(x, (uint64_t)R * k.tr), block_of(x, (uint64_t)C * k.tc), R, C) : (int)(t % (uint64_t)world);
        if (owner != rank) continue;
      }
      uint32_t need = need_mask(x, rank, (uint64_t)C * k.tc, std::min<uint64_t>((uint64_t)(C + 1) * k.tc, k.n_qry));
      if (k.sym) need |= need_mask(x, rank, (uint64_t)R * k.tr, std::min<uint64_t>((uint64_t)(R + 1) * k.tr, k.n_ref));
      uint32_t key = 0;
      for (int b = 0; b < 32; ++b) if (need >> b & 1u) key = std::max<uint32_t>(key, 1 + arrival_pos(x, rank, b / N_CHUNKS, b % N_CHUNKS));
      v.push_back({make_uint2(R | (C << 16), need), key});
    }
  }
  // all-vs-all: tiles that read only my own rows first, then in the order the other members' chunks arrive (row-major
  // within each group).  ref x query stays row-major: the queries are few and arrive early, while a column-wise sweep
  // would stream my whole ref plane from HBM once per query tile column.
  if (k.sym) std::stable_sort(v.begin(), v.end(), [](const T &a, const T &b) { return a.key < b.key; });
  out.resize(v.size());
  for (size_t i = 0; i < v.size(); ++i) out[i] = v[i].e;
}

static TileKey tile_key(int world, int symmetric, int use_path, uint32_t hv_d, uint32_t n_ref, const uint32_t *qb) {
  TileKey k = {};
  k.sym = symmetric;
  k.path = use_path;
  k.hv_d = hv_d;
  k.n_ref = symmetric ? qb[world] : n_ref;
  k.n_qry = qb[world];
  if (use_path == HG_PATH_NARROW) hg_narrow_tile_shape(&k.tr, &k.tc); else hg_tc_tile_shape(&k.tr, &k.tc);
  for (int m = 0; m <= world; ++m) k.qb[m] = qb[m];
  return k;
}

// This member's tiles for kernel `use_path` (3: 256 x 256 tiles, 2: 256 x 128), cached while the shapes stay the same.
static void build_tiles(hg_peer *p, const ShardCall &a, int use_path) {
  const TileKey k = tile_key(p->world, a.symmetric, use_path, a.hv_d, a.n_ref_local, a.qb);
  if (p->tiles_valid && memcmp(&k, &p->tiles_key, sizeof(k)) == 0) return;
  p->tiles_key = k;
  p->tiles_valid = true;
  p->tiles_on_device = false;
  plan_tiles(k, p->world, p->rank, p->tiles);
}

// The plan above without a GPU (host logic only; tests): tiles_out receives (tile row | tile column << 16, need mask)
// pairs; *n_tiles the count (HG_E_CAPACITY if it exceeds cap).
extern "C" int hg_peer_plan_tiles(int world, int rank, int symmetric, int path, uint32_t hv_d, uint32_t n_ref_local,
                                  const uint32_t *qry_bounds, uint32_t *tiles_out, uint64_t cap, uint64_t *n_tiles) {
  if (!qry_bounds || !n_tiles || world < 1 || world > HG_MAX_PEERS || rank < 0 || rank >= world || (path != HG_PATH_TWO_LIMB && path != HG_PATH_NARROW) || hv_d == 0) {
    hg_set_error("hg_peer_plan_tiles: bad argument"); return HG_E_INVALID;
  }
  std::vector<uint2> v;
  plan_tiles(tile_key(world, symmetric, path, hv_d, n_ref_local, qry_bounds), world, rank, v);
  *n_tiles = v.size();
  if (v.size() > cap || (!tiles_out && !v.empty())) { hg_set_error("hg_peer_plan_tiles: %zu tiles", v.size()); return HG_E_CAPACITY; }
  for (size_t i = 0; i < v.size(); ++i) { tiles_out[2 * i] = v[i].x; tiles_out[2 * i + 1] = v[i].y; }
  return HG_OK;
}

// The exchange plan of member `rank` without a GPU (host logic only; tests): chunk_rows_out[0 .. HG_PUSH_CHUNKS] = the
// row boundaries of its chunks (unused chunks are empty), units_out = (chunk index or HG_PUSH_CHUNKS for the start
// set, destination mask) per push unit in sending order, *ring = 1 if rows go to ring neighbours only.
static void plan_units(const XPlan &x, int rank, bool have_rows, std::vector<std::pair<int, uint32_t>> &units) {
  units.clear();
  uint32_t all = 0;
  for (int m = 0; m < x.world; ++m) if (m != rank) all |= 1u << m;
  if (x.world > 1) units.push_back({HG_PUSH_START_SET, all});
  if (!have_rows || x.world == 1) return;
  // chunk by chunk, every chunk to all its destinations at once: one NVLink destination takes 100-250 GB/s from a
  // GPU's pusher warps, four or seven together about 500 GB/s (measured, DESIGN.md 5)
  const uint32_t dest = dest_mask(x, rank);
  for (int c = 0; c < x.n_chunks[rank]; ++c) units.push_back({c, dest});
}
extern "C" int hg_peer_plan_push(int world, int rank, int symmetric, int path, uint32_t hv_d, const uint32_t *qry_bounds,
                                 uint32_t chunk_rows_out[HG_PUSH_CHUNKS + 1], uint32_t *units_out, uint64_t cap, uint64_t *n_units,
                                 int *ring) {
  if (!qry_bounds || !n_units || !chunk_rows_out || world < 1 || world > HG_MAX_PEERS || rank < 0 || rank >= world || (path != HG_PATH_TWO_LIMB && path != HG_PATH_NARROW) || hv_d == 0) {
    hg_set_error("hg_peer_plan_push: bad argument"); return HG_E_INVALID;
  }
  const XPlan x = make_xplan(world, symmetric, path, hv_d, qry_bounds);
  for (int c = 0; c <= N_CHUNKS; ++c) chunk_rows_out[c] = chunk_lo(x, rank, c);
  std::vector<std::pair<int, uint32_t>> u;
  plan_units(x, rank, qry_bounds[rank + 1] > qry_bounds[rank], u);
  *n_units = u.size();
  if (ring) *ring = x.ring;
  if (u.size() > cap || (!units_out && !u.empty())) { hg_set_error("hg_peer_plan_push: %zu units", u.size()); return HG_E_CAPACITY; }
  for (size_t i = 0; i < u.size(); ++i) { units_out[2 * i] = (uint32_t)u[i].first; units_out[2 * i + 1] = u[i].second; }
  return HG_OK;
}

// every allocation of the call, before anything that waits for another member is enqueued (growing a scratch
// buffer synchronises the device); also builds this member's tile list for kernel `use_path`
static int shard_reserve(hg_peer *p, const ShardCall &a, int use_path) {
  hg_ctx *c = p->ctx;
  HG_CUDA(cudaSetDevice(c->device));
  void *x;
  int rc;
  if (!a.symmetric && a.n_ref_local) {
    if ((rc = hg_scratch(c, HG_S_REF_LIMBS, hg_tc_mat_bytes(a.n_ref_local, a.hv_d) + 1024, &x))) return rc;
    if ((rc = hg_scratch(c, HG_S_NARROW_META, hg_narrow_arrays_bytes(a.n_ref_local) + (uint64_t)hg_narrow_set_cap(a.n_ref_local) * 4 + 256, &x))) return rc;
  }
  if (p->world > 1) {
    build_tiles(p, a, use_path);
    const size_t bytes = p->tiles.size() * sizeof(uint2) + 256;
    if ((rc = hg_scratch(c, HG_S_TILES, bytes, &x))) return rc;
    if ((rc = hg_pinned(c, 2, bytes, &x))) return rc;
    if (!p->tiles_on_device) memcpy(x, p->tiles.data(), p->tiles.size() * sizeof(uint2));
  }
  return HG_OK;
}

// rows whose first element is `d_rows` are rows [row0, ...) of a matrix: the matrix's (virtual) first element
static const int16_t *matrix_base(const int16_t *d_rows, uint32_t row0, uint32_t hv_d) {
  return (const int16_t *)((uintptr_t)d_rows - (uintptr_t)row0 * hv_d * 2);
}

// use_path 3: single s8 plane; 2: two s8 limb planes.  Enqueues everything on the member's stream; returns without waiting.
static int shard_enqueue(hg_peer *p, const ShardCall &a, int use_path) {
  hg_ctx *c = p->ctx;
  HG_CUDA(cudaSetDevice(c->device));
  int rc;
  const int rank = p->rank, world = p->world;
  const uint32_t n_total = a.qb[world], r0 = a.qb[rank], nl = a.qb[rank + 1] - a.qb[rank];
  uint8_t *W = p->win[rank];
  const ShardLayout lay = make_layout(world, n_total, a.hv_d, a.cap, use_path == HG_PATH_NARROW ? 1 : 2, a.mapped_hits != nullptr);
  int32_t *normW = (int32_t *)(W + lay.norm);
  // every member appends to ITS OWN list (local atomics and stores); peer_flush_kernel moves the list to the root afterwards
  hg_hit *hits = (hg_hit *)(W + OFF_HITS);
  unsigned long long *counter = (unsigned long long *)(W + OFF_COUNT);
  p->root = a.root;
  p->cap = a.cap;
  p->mapped_hits = a.mapped_hits;
  p->gather_off = lay.gather;
  c->ev_used &= ~(3 << 4);
  HG_PROF(c, 4);
  p->ev_n = 0;
  PEER_PROF(p, 0);
  // sequence number + 1, my hit counter and statistics reset, the root's gather counter reset
  peer_tick_kernel<<<1, 32, 0, c->stream>>>(W, rank, rank == a.root, use_path == HG_PATH_NARROW ? (uint32_t)rank * lay.set_cap : 0u, p->timeline);
  c->launches++;
  HG_CUDA(cudaGetLastError());
  hg_tile_feed feed = {};
  const bool use_list = world > 1;
  if (use_list) {
    if (!p->tiles_on_device) {
      HG_CUDA(cudaMemcpyAsync(c->d_scratch[HG_S_TILES], c->h_pinned[2], p->tiles.size() * sizeof(uint2), cudaMemcpyHostToDevice, c->stream));
      p->tiles_on_device = true;
    }
    feed.list = (const uint2 *)c->d_scratch[HG_S_TILES];
    feed.n_list = (uint32_t)p->tiles.size();
    feed.ready = (const uint32_t *)(W + OFF_READY);
    feed.seq_ptr = (const uint32_t *)(W + OFF_SEQ);
    feed.status = (uint32_t *)(W + OFF_STATUS);
    feed.timeout_ns = p->timeout_ns;
    feed.dbg = p->timeline ? reinterpret_cast<unsigned long long *>(W + OFF_DBG) : nullptr;
    // every other member's start set has landed: its pre-pass statistics and outlier entries (single plane), and - the
    // root raises its start flag after its tick kernel, in stream order - the root has reset its gather counter
    feed.start = (const uint32_t *)(W + OFF_START);
    for (int m = 0; m < world; ++m) if (m != rank) feed.start_need |= 1u << m;
  }
  if (nl) HG_CUDA(cudaMemcpyAsync(normW + r0, a.d_qry_norm, (size_t)nl * 4, cudaMemcpyDeviceToDevice, c->stream));
  hg_narrow_mat Qn, Rn;
  hg_tc_mat Qt, Rt;
  if (use_path == HG_PATH_NARROW) {
    if ((rc = hg_narrow_attach(c, matrix_base(a.d_qry_hv, r0, a.hv_d), n_total, a.hv_d, (int8_t *)(W + lay.plane), W + lay.arrays,
                               (uint32_t *)(W + lay.entries), (uint32_t *)(W + OFF_STATS_Q), (uint32_t)world, (uint32_t)rank,
                               (uint32_t)rank * lay.set_cap, lay.set_cap, &Qn, /*init_stats=*/false)))
      return rc;
    if ((rc = hg_narrow_prep_rows(c, &Qn, r0, nl))) return rc;
    if (!a.symmetric) {  // my own ref rows stay local; only their statistics are shared (the verdict must be the same everywhere)
      void *plane = c->d_scratch[HG_S_REF_LIMBS], *meta = c->d_scratch[HG_S_NARROW_META];
      const uint32_t nr = a.n_ref_local;
      if ((rc = hg_narrow_attach(c, a.d_ref_hv, nr, a.hv_d, (int8_t *)plane, meta, (uint32_t *)((uint8_t *)meta + hg_narrow_arrays_bytes(nr)),
                                 (uint32_t *)(W + OFF_STATS_R), (uint32_t)world, (uint32_t)rank, 0, hg_narrow_set_cap(nr), &Rn, /*init_stats=*/false)))
        return rc;
      if ((rc = hg_narrow_prep_rows(c, &Rn, 0, nr))) return rc;
    }
  } else {
    if ((rc = hg_tensor_shape_ok(a.hv_d, a.d_qry_hv, a.d_ref_hv))) return rc;
    if ((rc = hg_tc_attach(c, matrix_base(a.d_qry_hv, r0, a.hv_d), n_total, a.hv_d, (int8_t *)(W + lay.plane), &Qt))) return rc;
    if ((rc = hg_tc_split_rows(c, &Qt, r0, nl))) return rc;
    if (!a.symmetric && a.n_ref_local) {
      if ((rc = hg_tc_attach(c, a.d_ref_hv, a.n_ref_local, a.hv_d, (int8_t *)c->d_scratch[HG_S_REF_LIMBS], &Rt))) return rc;
      if ((rc = hg_tc_split_rows(c, &Rt, 0, a.n_ref_local))) return rc;
    }
  }
  PEER_PROF(p, 1);
  // ---- what I push to the others (hg_push_plan): the start set to everybody, then my rows chunk by chunk to the members
  //      that compute with them.  The dist kernel below carries pusher warps that do it while the tiles are computed; a
  //      member without a tile to compute pushes with stand-alone kernels instead ----
  const XPlan xp = make_xplan(world, a.symmetric, use_path, a.hv_d, a.qb);
  p->last_ring = xp.ring;
  hg_push_plan plan = {};
  for (int m = 0; m < world; ++m) plan.win[m] = p->win[m];
  plan.rank = rank;
  plan.world = world;
  plan.done = reinterpret_cast<uint32_t *>(W + OFF_DONE);
  plan.ready_off = OFF_READY;
  plan.start_off = OFF_START;
  plan.seq = (const uint32_t *)(W + OFF_SEQ);
  plan.dbg = p->timeline ? reinterpret_cast<unsigned long long *>(W + OFF_DBG) : nullptr;
  auto add = [&](int set, uint64_t off, uint64_t bytes) {
    if (bytes) { plan.off[set][plan.n[set]] = off; plan.bytes[set][plan.n[set]] = (uint32_t)bytes; plan.n[set]++; }
  };
  for (int ch = 0; ch < xp.n_chunks[rank] && world > 1; ++ch) {
    const uint64_t lo = chunk_lo(xp, rank, ch), n = chunk_lo(xp, rank, ch + 1) - lo;
    add(ch, lay.norm + lo * 4, n * 4);
    add(ch, lay.plane + lo * a.hv_d, n * a.hv_d);
    if (use_path == HG_PATH_NARROW) for (int k = 0; k < 5; ++k) add(ch, lay.arrays + ((uint64_t)k * n_total + lo) * 4, n * 4);
    else {
      add(ch, lay.plane + ((uint64_t)n_total + lo) * a.hv_d, n * a.hv_d);
      add(ch, lay.plane + 2 * (uint64_t)n_total * a.hv_d + lo * 8, n * 8);  // their row sums (hg_tc_mat::sq)
    }
  }
  if (use_path == HG_PATH_NARROW && world > 1) {  // the statistics and the outlier entries of ALL my rows (the pre-pass above is complete)
    if (nl) {  // (range 0 of the start set: the pushers cut it down to the entries the pre-pass actually wrote)
      add(HG_PUSH_START_SET, lay.entries + (uint64_t)rank * lay.set_cap * 4, (uint64_t)lay.set_cap * 4);
      plan.dyn_count = (const uint32_t *)(W + OFF_STATS_Q) + 4 * rank + 2;
      plan.dyn_base = (uint32_t)rank * lay.set_cap;
    }
    add(HG_PUSH_START_SET, OFF_STATS_Q + 16 * (uint64_t)rank, 16);
    if (!a.symmetric) add(HG_PUSH_START_SET, OFF_STATS_R + 16 * (uint64_t)rank, 16);
  }
  {
    std::vector<std::pair<int, uint32_t>> units;
    plan_units(xp, rank, nl > 0, units);
    plan.n_units = (int)units.size();
    for (int u = 0; u < plan.n_units; ++u) {
      plan.unit_set[u] = (uint8_t)units[u].first;
      plan.unit_dest[u] = (uint8_t)units[u].second;
      plan.unit_stamp[u] = -1;
    }
    // timeline: [8] start set out, [9] my first chunk at its first destination, [10] all chunks at the first destination, [11] all out
    if (plan.n_units > 0) plan.unit_stamp[0] = 8;
    if (plan.n_units > 1) { plan.unit_stamp[1] = 9; plan.unit_stamp[plan.n_units - 1] = 11; }
  }
  // Who pushes?  A member with tiles to compute: the pusher warps inside its dist kernel - one kernel computes tiles and
  // moves operands, no SM is given up.  A member without a tile to compute: stand-alone push kernels on its stream, ahead
  // of the dist launch (which then has nothing to do).
  const bool have_tiles = world > 1 && !p->tiles.empty() && (a.symmetric || a.n_ref_local > 0);
  if (world > 1 && !have_tiles) {
    for (int u = 0; u < plan.n_units; ++u) {
      const int set = plan.unit_set[u];
      PushArgs pa;
      pa.n = plan.n[set];
      for (int k = 0; k < pa.n; ++k) { pa.r[k].off = plan.off[set][k]; pa.r[k].bytes = plan.bytes[set][k]; }
      const uint64_t flag_off = set == HG_PUSH_START_SET ? OFF_START + 4 * (uint64_t)rank : OFF_READY + 4 * (uint64_t)(rank * N_CHUNKS + set);
      if ((rc = peer_push(p, pa, plan.unit_dest[u], flag_off, u))) return rc;
    }
  }
  const hg_push_plan *pp = have_tiles ? &plan : nullptr;
  PEER_PROF(p, 2);
  const hg_tile_feed *fp = use_list ? &feed : nullptr;
  if (use_path == HG_PATH_NARROW) {
    if (a.symmetric)
      rc = hg_narrow_launch_ex(c, &Qn, 0, n_total, 0, normW, &Qn, 0, n_total, 0, normW, a.ksize, a.ani_th, 1, hits, a.cap, counter, 1, 0, fp, pp);
    else
      rc = hg_narrow_launch_ex(c, &Rn, 0, a.n_ref_local, a.ref_row0, a.d_ref_norm, &Qn, 0, n_total, 0, normW, a.ksize, a.ani_th, 0, hits,
                               a.cap, counter, 1, 0, fp, pp);
  } else {
    if (a.symmetric)
      rc = hg_tc_launch_ex(c, &Qt, 0, n_total, 0, normW, &Qt, 0, n_total, 0, normW, a.ksize, a.ani_th, 1, hits, a.cap, counter, 1, 0, fp, pp);
    else
      rc = hg_tc_launch_ex(c, &Rt, 0, a.n_ref_local, a.ref_row0, a.d_ref_norm, &Qt, 0, n_total, 0, normW, a.ksize, a.ani_th, 0, hits, a.cap,
                           counter, 1, 0, fp, pp);
  }
  if (rc) return rc;
  HG_PROF(c, 5);
  PEER_PROF(p, 3);
  {  // my hits to the root: its gather list (NVLink), or the host buffer every member has mapped (my own PCIe link)
    hg_hit *dst = a.mapped_hits ? a.mapped_hits : (hg_hit *)(p->win[a.root] + lay.gather);
    unsigned long long *total = (unsigned long long *)(p->win[a.root] + OFF_TOTAL);
    peer_flush_kernel<<<64, 256, 0, c->stream>>>(W, total, dst, a.cap, p->timeline);
    c->launches++;
    HG_CUDA(cudaGetLastError());
  }
  if ((rc = peer_barrier(p))) return rc;  // every member has flushed: the root's list is complete, the windows may be reused
  HG_CUDA(cudaMemcpyAsync(p->h_hdr, W + OFF_STATUS, 128, cudaMemcpyDeviceToHost, c->stream));  // status word + hit counters
  PEER_PROF(p, 4);
  return HG_OK;
}

// Measurement support (with hg_set_profiling on the member's context): device ms of the last sharded dist's stages -
// [0] operands (pre-pass / limb split), [1] chunked push to the peers, [2] dist kernel (incl. its waits for the peers'
// chunks), [3] final barrier (wait for the slowest member).  Synchronises the member's stream.
extern "C" int hg_peer_stage_ms(hg_peer *p, float out_ms[4]) {
  if (!p || !out_ms) { hg_set_error("hg_peer_stage_ms: NULL argument"); return HG_E_INVALID; }
  HG_CUDA(cudaSetDevice(p->ctx->device));
  HG_CUDA(cudaStreamSynchronize(p->ctx->stream));
  for (int i = 0; i < 4; ++i) {
    out_ms[i] = -1.0f;
    if (p->ev_n >= i + 2) HG_CUDA(cudaEventElapsedTime(&out_ms[i], p->ev[i], p->ev[i + 1]));
  }
  return HG_OK;
}

// Measurement support (HG_PEER_TIMELINE=1 in the environment when the group is created): globaltimer stamps (ns) of the
// last sharded dist on this member - [0] first node, [1] dist kernel entry, [2] start flags seen, [3] ns CTA 0's producer
// waited for rows, [4] last CTA done, [5] longest producer wait, [8..11] my chunk c pushed, [12] hit flush, [13] barrier
// entry, [14] barrier exit, [16] barrier exit of the call before (all members leave a barrier within about a microsecond:
// the common time base).  Synchronises the member's stream.
extern "C" int hg_peer_timeline(hg_peer *p, unsigned long long out[32]) {
  if (!p || !out) { hg_set_error("hg_peer_timeline: NULL argument"); return HG_E_INVALID; }
  HG_CUDA(cudaSetDevice(p->ctx->device));
  HG_CUDA(cudaStreamSynchronize(p->ctx->stream));
  HG_CUDA(cudaMemcpy(out, p->win[p->rank] + OFF_DBG, 32 * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
  return HG_OK;
}

static int peer_status(hg_peer *p) {  // after a stream synchronisation that followed a sharded dist (h_hdr is current)
  if (*reinterpret_cast<const uint32_t *>(p->h_hdr)) {
    cudaMemset(p->win[p->rank] + OFF_STATUS, 0, 4);
    *reinterpret_cast<uint32_t *>(p->h_hdr) = 0;
    hg_set_error("a member of the GPU group did not deliver its rows / reach a barrier within %llu ms", p->timeout_ns / 1000000ull);
    return HG_E_CUDA;
  }
  return HG_OK;
}

// verdict of the single-plane pre-passes of ALL members (their statistics were pushed into every window, so every
// member reads the same answer): HG_OK narrow, HG_E_UNSUPPORTED not narrow (*absmax = max |hv| over all rows)
static int shard_verdict(hg_peer *p, const ShardCall &a, int32_t *absmax) {
  hg_ctx *c = p->ctx;
  uint32_t sq[4 * HG_MAX_PEERS], sr[4 * HG_MAX_PEERS];
  HG_CUDA(cudaMemcpyAsync(sq, p->win[p->rank] + OFF_STATS_Q, sizeof(sq), cudaMemcpyDeviceToHost, c->stream));
  HG_CUDA(cudaMemcpyAsync(sr, p->win[p->rank] + OFF_STATS_R, sizeof(sr), cudaMemcpyDeviceToHost, c->stream));
  HG_CUDA(cudaStreamSynchronize(c->stream));
  int rc = peer_status(p);
  if (rc) return rc;
  uint32_t declined = 0, amax = 0;
  for (int r = 0; r < p->world; ++r) {
    declined |= sq[4 * r + 3];
    amax = std::max(amax, sq[4 * r]);
    if (!a.symmetric) { declined |= sr[4 * r + 3]; amax = std::max(amax, sr[4 * r]); }
  }
  *absmax = (int32_t)amax;
  return declined ? HG_E_UNSUPPORTED : HG_OK;
}

static void shard_reason(hg_peer *p, int path, int32_t absmax, bool forced) {
  hg_ctx *c = p->ctx;
  if (path == HG_PATH_NARROW)
    hg_dist_record(c, path, "tensor-narrow%s: member %d of %d GPUs, operand planes pushed over NVLink windows in chunks, %s, tiles ordered by arrival%s",
             forced ? " (forced)" : "", p->rank, p->world, p->last_ring ? "block pairs owned along the ring (rows go to N/2 members)" : "tiles dealt round-robin (rows go to every member)",
             forced ? "" : "; rows fit one s8 plane as x = 2a + s");
  else
    hg_dist_record(c, path, "tensor%s: member %d of %d GPUs, two s8 limb planes pushed over NVLink windows in chunks, %s, tiles ordered by arrival (max |hv| = %d)",
             forced ? " (forced)" : "", p->rank, p->world, p->last_ring ? "block pairs owned along the ring (rows go to N/2 members)" : "tiles dealt round-robin (rows go to every member)", absmax);
}

// Collective over the group (every member calls it with the same scalars and its own rows); see hypergen_b200.h.
extern "C" int hg_dist_sharded_dev(hg_peer *p, const int16_t *d_ref_hv, const int32_t *d_ref_norm2, uint32_t n_ref_local,
                                   uint32_t ref_row0, const int16_t *d_qry_hv, const int32_t *d_qry_norm2, const uint32_t *qry_bounds,
                                   uint32_t hv_d, uint32_t ksize, float ani_th, int symmetric, int path, int root, uint64_t cap,
                                   hg_hit *mapped_hits) {
  if (!p || !qry_bounds) { hg_set_error("hg_dist_sharded_dev: NULL argument"); return HG_E_INVALID; }
  ShardCall a = {};
  a.d_ref_hv = d_ref_hv; a.d_ref_norm = d_ref_norm2; a.n_ref_local = symmetric ? 0u : n_ref_local; a.ref_row0 = ref_row0;
  a.d_qry_hv = d_qry_hv; a.d_qry_norm = d_qry_norm2;
  for (int m = 0; m <= p->world; ++m) a.qb[m] = qry_bounds[m];
  a.hv_d = hv_d; a.ksize = ksize; a.ani_th = ani_th; a.symmetric = symmetric; a.root = root; a.cap = cap; a.mapped_hits = mapped_hits;
  int rc;
  if ((rc = shard_check(p, a))) return rc;
  if (path != HG_PATH_AUTO && path != HG_PATH_TWO_LIMB && path != HG_PATH_NARROW) { hg_set_error("hg_dist_sharded_dev: path %d (0 auto, 2 two-limb, 3 single plane)", path); return HG_E_INVALID; }
  if (a.qb[p->world] == 0) return HG_OK;
  if (path == HG_PATH_TWO_LIMB || path == HG_PATH_NARROW) {
    if (path == HG_PATH_NARROW && (rc = hg_tensor_shape_ok(hv_d, d_qry_hv, d_ref_hv))) return rc;
    hg_ctx *c = p->ctx;
    // The same call again (same pointers, shapes and scratch buffers): replay its launch sequence as a CUDA graph.
    // The first call runs directly, the second is captured, the following ones are one cudaGraphLaunch each.
    std::vector<uint8_t> key(sizeof(ShardCall) + 4 * sizeof(void *));
    memcpy(key.data(), &a, sizeof(ShardCall));
    const void *extra[4] = {c->d_scratch[HG_S_REF_LIMBS], c->d_scratch[HG_S_NARROW_META], c->d_scratch[HG_S_TILES], (const void *)(uintptr_t)path};
    memcpy(key.data() + sizeof(ShardCall), extra, sizeof(extra));
    const bool can_graph = !c->prof && !getenv("HG_PEER_NO_GRAPH");
    if (can_graph && p->graph && key == p->graph_key) {
      HG_CUDA(cudaSetDevice(c->device));
      HG_CUDA(cudaGraphLaunch(p->graph, c->stream));
      c->launches += p->graph_nodes;
      shard_reason(p, path, -1, true);
      return HG_OK;
    }
    if (p->graph) { cudaGraphExecDestroy(p->graph); p->graph = nullptr; p->graph_key.clear(); }
    if ((rc = shard_reserve(p, a, path))) return rc;
    memcpy(key.data() + sizeof(ShardCall), extra, 0);  // (scratch pointers may have changed in shard_reserve: refresh below)
    const void *extra2[4] = {c->d_scratch[HG_S_REF_LIMBS], c->d_scratch[HG_S_NARROW_META], c->d_scratch[HG_S_TILES], (const void *)(uintptr_t)path};
    memcpy(key.data() + sizeof(ShardCall), extra2, sizeof(extra2));
    if (can_graph && key == p->last_key && p->tiles_on_device) {
      HG_CUDA(cudaSetDevice(c->device));
      const unsigned long long l0 = c->launches;
      cudaGraph_t g = nullptr;
      HG_CUDA(cudaStreamBeginCapture(c->stream, cudaStreamCaptureModeThreadLocal));
      rc = shard_enqueue(p, a, path);
      const cudaError_t e = cudaStreamEndCapture(c->stream, &g);
      if (rc) { if (g) cudaGraphDestroy(g); return rc; }
      if (e != cudaSuccess) return hg_cuda_fail(e, "cudaStreamEndCapture", __FILE__, __LINE__);
      const cudaError_t e2 = cudaGraphInstantiate(&p->graph, g, 0);
      cudaGraphDestroy(g);
      if (e2 != cudaSuccess) { p->graph = nullptr; return hg_cuda_fail(e2, "cudaGraphInstantiate", __FILE__, __LINE__); }
      p->graph_key = key;
      p->graph_nodes = (unsigned)(c->launches - l0);
      HG_CUDA(cudaGraphLaunch(p->graph, c->stream));
    } else {
      if ((rc = shard_enqueue(p, a, path))) return rc;
      p->last_key = key;
    }
    shard_reason(p, path, -1, true);
    return HG_OK;
  }
  int32_t absmax = -1;
  if (p->graph) { cudaGraphExecDestroy(p->graph); p->graph = nullptr; p->graph_key.clear(); }
  p->last_key.clear();
  rc = hg_tensor_shape_ok(hv_d, d_qry_hv, d_ref_hv);
  if (rc == HG_OK) {
    if ((rc = shard_reserve(p, a, HG_PATH_NARROW))) return rc;
    if ((rc = shard_enqueue(p, a, HG_PATH_NARROW))) return rc;
    rc = shard_verdict(p, a, &absmax);
    if (rc == HG_OK) { shard_reason(p, HG_PATH_NARROW, absmax, false); return HG_OK; }
    if (rc != HG_E_UNSUPPORTED) return rc;
  }
  if (absmax > HG_LIMB_MAX_ABS) {
    hg_set_error("hg_dist_sharded_dev: max |hv| = %d exceeds the 13-bit budget of the int8 limb split; the sharded path has no SIMT kernel", absmax);
    return HG_E_UNSUPPORTED;
  }
  if ((rc = shard_reserve(p, a, HG_PATH_TWO_LIMB))) return rc;
  if ((rc = shard_enqueue(p, a, HG_PATH_TWO_LIMB))) return rc;
  shard_reason(p, HG_PATH_TWO_LIMB, absmax, false);
  return HG_OK;
}

// After hg_dist_sharded_dev: waits for this member's stream.  On the root: the number of hits (HG_E_CAPACITY with the
// need if it exceeds cap), the hits - in dump_ani_file's order if `sorted` (ani_milli as hg_dist_sorted) - copied to
// HOST memory.  On the other members: n_hits = 0 (hits may be NULL).
extern "C" int hg_dist_sharded_hits(hg_peer *p, int sorted, hg_hit *hits, uint32_t *ani_milli, uint64_t cap, uint64_t *n_hits) {
  if (!p || !n_hits) { hg_set_error("hg_dist_sharded_hits: NULL argument"); return HG_E_INVALID; }
  hg_ctx *c = p->ctx;
  *n_hits = 0;
  HG_CUDA(cudaSetDevice(c->device));
  int rc;
  HG_CUDA(cudaStreamSynchronize(c->stream));
  const unsigned long long cnt =  // written by the call's last node
      p->rank == p->root ? *reinterpret_cast<const unsigned long long *>(p->h_hdr + (OFF_TOTAL - OFF_STATUS)) : 0ull;
  if ((rc = peer_status(p))) return rc;
  if (p->rank != p->root) return HG_OK;
  *n_hits = cnt;
  if (cnt > cap || cnt > p->cap) {
    hg_set_error("hg_dist_sharded: %llu pairs pass the threshold, capacity is %llu", cnt, (unsigned long long)std::min<uint64_t>(cap, p->cap));
    return HG_E_CAPACITY;
  }
  if (cnt == 0) return HG_OK;
  if (p->mapped_hits) {  // the kernels wrote the records into the caller's mapped host buffer: nothing to copy
    if (sorted) { hg_set_error("hg_dist_sharded_hits: hits in a mapped host buffer are not sorted on the device"); return HG_E_UNSUPPORTED; }
    return HG_OK;
  }
  if (!hits) { hg_set_error("hg_dist_sharded_hits: hits is NULL"); return HG_E_INVALID; }
  return hg_hits_to_host(c, (hg_hit *)(p->win[p->rank] + p->gather_off), cnt, sorted != 0, hits, ani_milli);
}

// device pointers of the root's hit list and counter as this member addresses them (benchmarks, callers with their own tail)
extern "C" int hg_peer_hit_buffers(hg_peer *p, int root, hg_hit **d_hits, unsigned long long **d_count) {
  if (!p || root < 0 || root >= p->world || !p->connected) { hg_set_error("hg_peer_hit_buffers: bad argument"); return HG_E_INVALID; }
  if (d_hits) *d_hits = (hg_hit *)(p->win[root] + p->gather_off);
  if (d_count) *d_count = (unsigned long long *)(p->win[root] + OFF_TOTAL);
  return HG_OK;
}

// ---------------------------------------------------------------------------------------------------
// one process, all the GPUs of the box: what `hyper-gen sketch -D gpu` / `hyper-gen dist` call
// (the reference is single-GPU: CudaDevice::new(0), src/sketch_cuda.rs:52)
// ---------------------------------------------------------------------------------------------------
struct hg_group {
  int n;
  hg_ctx *ctx[HG_MAX_PEERS];
  hg_peer *peer[HG_MAX_PEERS];
  uint64_t window_bytes;
};

extern "C" int hg_group_create(int n_devices, const int *ordinals, hg_group **out) {
  if (!out) { hg_set_error("hg_group_create: out is NULL"); return HG_E_INVALID; }
  *out = nullptr;
  int avail = 0;
  cudaError_t e = cudaGetDeviceCount(&avail);
  if (e != cudaSuccess || avail == 0) {
    hg_set_error("hg_group_create: no CUDA device (%s); this library has no CPU fallback", e == cudaSuccess ? "device count 0" : cudaGetErrorString(e));
    return HG_E_CUDA;
  }
  if (n_devices <= 0) n_devices = std::min(avail, HG_MAX_PEERS);  // all visible GPUs
  if (n_devices > HG_MAX_PEERS) { hg_set_error("hg_group_create: at most %d devices", HG_MAX_PEERS); return HG_E_INVALID; }
  hg_group *g = new hg_group();
  memset(g, 0, sizeof(*g));
  g->n = n_devices;
  for (int i = 0; i < n_devices; ++i) {
    const int rc = hg_init(ordinals ? ordinals[i] : i, &g->ctx[i]);
    if (rc) { hg_group_destroy(g); return rc; }
  }
  *out = g;
  return HG_OK;
}

extern "C" void hg_group_destroy(hg_group *g) {
  if (!g) return;
  for (int i = 0; i < g->n; ++i) if (g->peer[i]) hg_peer_destroy(g->peer[i]);
  for (int i = 0; i < g->n; ++i) if (g->ctx[i]) hg_destroy(g->ctx[i]);
  delete g;
}

extern "C" int hg_group_size(const hg_group *g) { return g ? g->n : 0; }
extern "C" hg_ctx *hg_group_ctx(hg_group *g, int i) { return g && i >= 0 && i < g->n ? g->ctx[i] : nullptr; }

static int group_windows(hg_group *g, uint64_t need) {
  if (g->peer[0] && g->window_bytes >= need) return HG_OK;
  for (int i = 0; i < g->n; ++i) if (g->peer[i]) { hg_peer_destroy(g->peer[i]); g->peer[i] = nullptr; }
  need += need / 8;
  int rc = hg_peer_create_local(g->ctx, g->n, need, g->peer);
  if (rc) return rc;
  g->window_bytes = need;
  return HG_OK;
}

// contiguous split of n items with weights w[i] = off[i + 1] - off[i] into `parts` runs of about equal weight
static std::vector<uint32_t> split_by_weight(const uint64_t *off, uint32_t n, int parts) {
  std::vector<uint32_t> b(parts + 1, n);
  b[0] = 0;
  const uint64_t total = off[n] - off[0];
  uint32_t g = 0;
  for (int k = 1; k < parts; ++k) {
    const uint64_t target = off[0] + total / parts * k + (total % parts) * k / parts;
    while (g < n && off[g + 1] - (off[g + 1] - off[g]) / 2 <= target) ++g;  // an item goes where its midpoint falls
    b[k] = g;
  }
  return b;
}

// hg_sketch_fasta_batch over all GPUs of the group: the files are split into one contiguous run per GPU of about
// equal bytes (genomes are independent - no collective, SURVEY.md §8e); one host thread per GPU drives its pipeline.
extern "C" int hg_group_sketch_fasta_batch(hg_group *g, const uint8_t *raw, const uint64_t *file_off, uint32_t n_files,
                                           const hg_sketch_params *p, int16_t *hv, uint8_t *packed, uint8_t *quant_bits,
                                           int32_t *norm2, uint32_t *n_hashes) {
  if (!g || !file_off || !p) { hg_set_error("hg_group_sketch_fasta_batch: NULL argument"); return HG_E_INVALID; }
  if (n_files == 0) return HG_OK;
  for (uint32_t f = 0; f < n_files; ++f)
    if (file_off[f + 1] < file_off[f]) { hg_set_error("file_off not monotone at %u", f); return HG_E_INVALID; }
  const int parts = (int)std::min<uint32_t>((uint32_t)g->n, n_files);
  const std::vector<uint32_t> b = split_by_weight(file_off, n_files, parts);
  std::vector<int> rcs(parts, HG_OK);
  std::vector<std::string> msgs(parts);
  std::vector<std::thread> th;
  const uint32_t D = p->hv_d;
  for (int k = 0; k < parts; ++k) {
    th.emplace_back([&, k]() {
      const uint32_t f0 = b[k], m = b[k + 1] - b[k];
      if (m == 0) return;
      rcs[k] = hg_sketch_fasta_batch(g->ctx[k], raw, file_off + f0, m, p, hv ? hv + (size_t)f0 * D : nullptr,
                                     packed ? packed + (size_t)f0 * 2 * D : nullptr, quant_bits ? quant_bits + f0 : nullptr,
                                     norm2 ? norm2 + f0 : nullptr, n_hashes ? n_hashes + f0 : nullptr);
      if (rcs[k]) msgs[k] = hg_last_error();
    });
  }
  for (auto &t : th) t.join();
  for (int k = 0; k < parts; ++k)
    if (rcs[k]) { hg_set_error("GPU %d (files %u..%u): %s", g->ctx[k]->device, b[k], b[k + 1], msgs[k].c_str()); return rcs[k]; }
  return HG_OK;
}

// hg_sketch_fasta_records over all GPUs of the group: the files split as above.  Each member sketches its run and keeps
// the rows on its device; once the total is known to fit rec_cap, each member copies its rows to its prefix offset.
extern "C" int hg_group_sketch_fasta_records(hg_group *g, const uint8_t *raw, const uint64_t *file_off, uint32_t n_files,
                                             const hg_sketch_params *p, uint32_t rec_cap, hg_fasta_record *records,
                                             uint8_t *packed, uint8_t *quant_bits, int32_t *norm2, uint32_t *n_hashes,
                                             uint32_t *n_records) {
  if (!g || !file_off || !p || !n_records) { hg_set_error("hg_group_sketch_fasta_records: NULL argument"); return HG_E_INVALID; }
  *n_records = 0;
  if (n_files == 0) return HG_OK;
  if (!raw && file_off[n_files] > file_off[0]) { hg_set_error("hg_group_sketch_fasta_records: raw is NULL"); return HG_E_INVALID; }
  for (uint32_t f = 0; f < n_files; ++f)
    if (file_off[f + 1] < file_off[f]) { hg_set_error("file_off not monotone at %u", f); return HG_E_INVALID; }
  const int parts = (int)std::min<uint32_t>((uint32_t)g->n, n_files);
  const std::vector<uint32_t> b = split_by_weight(file_off, n_files, parts);
  std::vector<hg_records_part> part(parts);
  std::vector<int> rcs(parts, HG_OK);
  std::vector<std::string> msgs(parts);
  auto run_all = [&](const std::function<int(int)> &fn) {  // one host thread per member with files
    std::vector<std::thread> th;
    for (int k = 0; k < parts; ++k)
      if (b[k + 1] > b[k])
        th.emplace_back([&, k]() {
          rcs[k] = fn(k);
          if (rcs[k]) msgs[k] = hg_last_error();
        });
    for (auto &t : th) t.join();
    for (int k = 0; k < parts; ++k)
      if (rcs[k]) { hg_set_error("GPU %d (files %u..%u): %s", g->ctx[k]->device, b[k], b[k + 1], msgs[k].c_str()); return rcs[k]; }
    return (int)HG_OK;
  };
  int rc = run_all([&](int k) { return hg_records_run(g->ctx[k], raw, file_off + b[k], b[k + 1] - b[k], p, rec_cap, part[k]); });
  if (rc) return rc;
  std::vector<uint64_t> pre(parts + 1, 0);
  for (int k = 0; k < parts; ++k) pre[k + 1] = pre[k] + part[k].rec.size();
  if (pre[parts] > 0xFFFFFFFFull) { hg_set_error("more than 2^32 - 1 records in one call"); return HG_E_UNSUPPORTED; }
  *n_records = (uint32_t)pre[parts];
  if (pre[parts] > rec_cap) {
    hg_set_error("hg_group_sketch_fasta_records: %u records, rec_cap is %u", *n_records, rec_cap);
    return HG_E_CAPACITY;
  }
  const size_t D = p->hv_d;
  return run_all([&](int k) {
    const uint64_t r0 = pre[k];
    if (records)
      for (size_t r = 0; r < part[k].rec.size(); ++r) {
        records[r0 + r] = part[k].rec[r];
        records[r0 + r].file += b[k];
      }
    return hg_records_fetch(g->ctx[k], part[k], p->hv_d, packed ? packed + r0 * 2 * D : nullptr, quant_bits ? quant_bits + r0 : nullptr,
                            norm2 ? norm2 + r0 : nullptr, n_hashes ? n_hashes + r0 : nullptr);
  });
}

// hg_dist_packed over all GPUs of the group.  Every GPU receives a contiguous block of the packed ref rows and of the
// packed query rows over its own PCIe link, unpacks them, and the sharded dist above does the rest; the hits come back
// from GPU 0 (sorted there if asked).  Same arguments and capacity contract as hg_dist_packed.
extern "C" int hg_group_dist_packed(hg_group *g, const uint8_t *ref_packed, uint64_t ref_stride, const uint8_t *ref_bits,
                                    const int32_t *ref_norm, uint32_t n_ref, const uint8_t *qry_packed, uint64_t qry_stride,
                                    const uint8_t *qry_bits, const int32_t *qry_norm, uint32_t n_qry, uint32_t hv_d,
                                    uint32_t ksize, float ani_th, int symmetric, int sorted, hg_hit *hits, uint32_t *ani_milli,
                                    uint64_t cap, uint64_t *n_hits) {
  if (!g || !n_hits) { hg_set_error("hg_group_dist_packed: NULL argument"); return HG_E_INVALID; }
  *n_hits = 0;
  hg_packed_rows R = {ref_packed, ref_stride, ref_bits, ref_norm, n_ref}, Q = {qry_packed, qry_stride, qry_bits, qry_norm, n_qry};
  int rc;
  if (cap && !hits) { hg_set_error("hg_group_dist_packed: NULL argument"); return HG_E_INVALID; }
  if ((rc = hg_packed_args_check("hg_group_dist_packed", R, Q, hv_d))) return rc;
  if (n_ref == 0 || n_qry == 0) return HG_OK;
  bool same;
  if ((rc = hg_packed_rows_check("hg_group_dist_packed", &R, &Q, hv_d, &same))) return rc;
  const uint32_t bmax = std::max(R.max_bits, Q.max_bits);
  // a single GPU, too little work to share, a shape only the single-GPU entry handles (one matrix against itself with
  // both orders, the j > i filter over two different matrices), or rows beyond the limb split (its exact SIMT kernel)
  if (g->n == 1 || (uint64_t)n_ref * n_qry < 1024ull * 1024ull || hv_d % 512 != 0 || (same && !symmetric) || (!same && symmetric) ||
      bmax > 13)
    return hg_dist_packed_run(g->ctx[0], R, Q, same, hv_d, ksize, ani_th, symmetric, HG_PATH_AUTO, sorted != 0, hits, ani_milli, cap,
                              n_hits);
  const int N = g->n;
  if ((rc = group_windows(g, hg_peer_window_need(n_qry, hv_d, cap)))) return rc;
  // row blocks: multiples of 256 rows when there are enough rows (what the ring ownership of the all-vs-all needs), else of 4
  auto bound = [&](uint32_t n, int k) -> uint32_t {
    if (k >= N) return n;
    if (n >= 512u * (uint32_t)N) return std::min<uint32_t>(n, 256u * (uint32_t)(((uint64_t)k * ((n + 255) / 256) + N / 2) / N));  // the 256-row tile rows, dealt evenly
    return (uint32_t)(((uint64_t)n * k / N) & ~3ull);
  };
  struct Member { uint32_t r0; HostRows r, q; };  // a self-comparison has no ref block: its query rows are all of it
  std::vector<Member> M(N);
  auto make_call = [&](const Member &m) {
    ShardCall a = {};
    a.d_ref_hv = m.r.d_hv; a.d_ref_norm = m.r.d_norm; a.n_ref_local = m.r.n; a.ref_row0 = m.r0;
    a.d_qry_hv = m.q.d_hv; a.d_qry_norm = m.q.d_norm;
    for (int k = 0; k <= N; ++k) a.qb[k] = bound(n_qry, k);
    a.hv_d = hv_d; a.ksize = ksize; a.ani_th = ani_th; a.symmetric = symmetric; a.root = 0; a.cap = cap; a.mapped_hits = nullptr;
    return a;
  };
  // phase 1: every allocation, on every GPU
  for (int k = 0; k < N; ++k) {
    hg_ctx *c = g->ctx[k];
    Member &m = M[k];
    const uint32_t q0 = bound(n_qry, k);
    m.r0 = same ? 0 : bound(n_ref, k);
    const uint32_t rn = same ? 0 : bound(n_ref, k + 1) - m.r0;
    HG_CUDA(cudaSetDevice(c->device));
    if ((rc = hg_packed_stage(c, R.rows(m.r0, rn), Q.rows(q0, bound(n_qry, k + 1) - q0), false, hv_d, &m.r, &m.q))) return rc;
    if ((rc = shard_check(g->peer[k], make_call(m)))) return rc;
  }
  // b-bit values are below 2^(b-1): above 10 bits no row fits the single plane, and up to 13 bits every element fits two limbs
  int used = bmax > 10 ? HG_PATH_TWO_LIMB : HG_PATH_NARROW;
  for (int k = 0; k < N; ++k)
    if ((rc = shard_reserve(g->peer[k], make_call(M[k]), used))) return rc;
  // phase 2: H2D + unpack + sharded dist enqueued on every GPU; nothing here waits for another GPU
  auto enqueue_all = [&](int use_path) -> int {
    for (int k = 0; k < N; ++k) {
      hg_ctx *c = g->ctx[k];
      Member &m = M[k];
      HG_CUDA(cudaSetDevice(c->device));
      int r2 = shard_enqueue(g->peer[k], make_call(m), use_path);
      if (r2) return r2;
    }
    return HG_OK;
  };
  for (int k = 0; k < N; ++k) {
    HG_CUDA(cudaSetDevice(g->ctx[k]->device));
    if ((rc = hg_rows_to_device(g->ctx[k], M[k].q, hv_d)) || (rc = hg_rows_to_device(g->ctx[k], M[k].r, hv_d))) return rc;
  }
  int32_t absmax = -1;
  if ((rc = enqueue_all(used))) return rc;
  if (used == HG_PATH_NARROW) {
    int verdict = HG_OK;
    for (int k = 0; k < N; ++k) {
      cudaSetDevice(g->ctx[k]->device);
      const int v = shard_verdict(g->peer[k], make_call(M[k]), &absmax);
      if (v != HG_OK && v != HG_E_UNSUPPORTED) return v;
      if (v) verdict = v;
    }
    if (verdict == HG_E_UNSUPPORTED) {  // not narrow (the same answer on every GPU): the two-limb kernel on the rows already in HBM
      used = HG_PATH_TWO_LIMB;
      for (int k = 0; k < N; ++k)
        if ((rc = shard_reserve(g->peer[k], make_call(M[k]), HG_PATH_TWO_LIMB))) return rc;
      if ((rc = enqueue_all(HG_PATH_TWO_LIMB))) return rc;
    }
  }
  for (int k = 0; k < N; ++k) shard_reason(g->peer[k], used, absmax, false);
  for (int k = N - 1; k >= 0; --k) {
    uint64_t nh = 0;
    rc = hg_dist_sharded_hits(g->peer[k], sorted, k == 0 ? hits : nullptr, k == 0 ? ani_milli : nullptr, cap, &nh);
    if (k == 0) *n_hits = nh;
    if (rc) return rc;
  }
  return HG_OK;
}

// hg_search_packed over all GPUs of the group (DESIGN.md §4.8).  The refs are cut into contiguous blocks of about equal
// size, one per member that gets at least 1024 of them; each member copies its ref block and all query rows over its own
// PCIe link and searches them.  One host thread per GPU drives its members: members that share a device ordinal run one
// after another (the dist kernels were never checked running next to another context's on the same GPU).  The blocks'
// results are copied to GPU 0 and merged there; the only exchange is n_qry * top_k records per member, so no windows.
extern "C" int hg_group_search_packed(hg_group *g, const uint8_t *ref_packed, uint64_t ref_stride, const uint8_t *ref_bits,
                                      const int32_t *ref_norm, uint32_t n_ref, const uint8_t *qry_packed, uint64_t qry_stride,
                                      const uint8_t *qry_bits, const int32_t *qry_norm, uint32_t n_qry, uint32_t hv_d, uint32_t ksize,
                                      uint32_t top_k, float ani_min, int path, hg_hit *out, uint32_t *n_found, uint32_t *ani_milli) {
  if (!g) { hg_set_error("hg_group_search_packed: NULL argument"); return HG_E_INVALID; }
  for (int k = 0; k < g->n; ++k) {  // a member without a block reports no passes
    memset(g->ctx[k]->search_stats, 0, sizeof(g->ctx[k]->search_stats));
    g->ctx[k]->search_ev_used = 0;
  }
  hg_packed_rows R = {ref_packed, ref_stride, ref_bits, ref_norm, n_ref}, Q = {qry_packed, qry_stride, qry_bits, qry_norm, n_qry};
  const char *who = "hg_group_search_packed";
  int rc;
  if ((rc = hg_packed_args_check(who, R, Q, hv_d)) || (rc = hg_search_check(who, n_qry, out, n_found, hv_d, top_k, path))) return rc;
  const int parts = (int)std::min<uint32_t>((uint32_t)g->n, std::max<uint32_t>(1u, n_ref / 1024u));
  if (parts == 1) return hg_search_packed_host(g->ctx[0], who, R, Q, hv_d, ksize, top_k, ani_min, path, out, n_found, ani_milli);
  if (n_qry == 0) return HG_OK;
  bool same;
  if ((rc = hg_packed_rows_check(who, &R, &Q, hv_d, &same))) return rc;
  std::vector<uint32_t> b(parts + 1);
  for (int k = 0; k <= parts; ++k) b[k] = (uint32_t)((uint64_t)n_ref * k / parts);
  std::vector<hg_hit *> d_out(parts);
  std::vector<uint32_t *> d_nf(parts), d_milli(parts);
  std::vector<int> rcs(parts, HG_OK);
  std::vector<std::string> msgs(parts);
  auto member = [&](int m) -> int {  // every member holds a ref block and all queries: two matrices, even when `same`
    hg_ctx *c = g->ctx[m];
    HG_CUDA(cudaSetDevice(c->device));
    return hg_search_packed_run(c, R.rows(b[m], b[m + 1] - b[m]), Q, false, hv_d, ksize, top_k, ani_min, path, &d_out[m], &d_nf[m],
                                &d_milli[m]);
  };
  std::vector<std::thread> th;
  for (int k = 0; k < parts; ++k) {
    bool first_on_device = true;
    for (int l = 0; l < k; ++l) first_on_device &= g->ctx[l]->device != g->ctx[k]->device;
    if (!first_on_device) continue;
    th.emplace_back([&, k]() {
      for (int m = k; m < parts; ++m) {
        if (g->ctx[m]->device != g->ctx[k]->device) continue;
        if ((rcs[m] = member(m))) msgs[m] = hg_last_error();
      }
    });
  }
  for (auto &t : th) t.join();
  for (int k = 0; k < parts; ++k)
    if (rcs[k]) { hg_set_error("GPU %d (refs %u..%u): %s", g->ctx[k]->device, b[k], b[k + 1], msgs[k].c_str()); return rcs[k]; }
  // gather: the members' results next to each other on GPU 0, in a slot apart from member 0's own result (HG_S_TILES)
  hg_ctx *c0 = g->ctx[0];
  HG_CUDA(cudaSetDevice(c0->device));
  const size_t n_out = (size_t)n_qry * top_k;
  void *d_gather, *d_res;
  if ((rc = hg_scratch(c0, HG_S_PACKED, (size_t)parts * (n_out * sizeof(hg_hit) + (size_t)n_qry * 4) + 256, &d_gather))) return rc;
  if ((rc = hg_scratch(c0, HG_S_SORT_TMP, n_out * (sizeof(hg_hit) + 4) + (size_t)n_qry * 4 + 256, &d_res))) return rc;
  hg_hit *g_hits = (hg_hit *)d_gather;
  uint32_t *g_found = (uint32_t *)(g_hits + (size_t)parts * n_out);
  for (int k = 0; k < parts; ++k) {
    const int dev = g->ctx[k]->device;
    HG_CUDA(cudaMemcpyPeerAsync(g_hits + (size_t)k * n_out, c0->device, d_out[k], dev, n_out * sizeof(hg_hit), c0->stream));
    HG_CUDA(cudaMemcpyPeerAsync(g_found + (size_t)k * n_qry, c0->device, d_nf[k], dev, (size_t)n_qry * 4, c0->stream));
  }
  hg_hit *r_out = (hg_hit *)d_res;
  uint32_t *r_milli = (uint32_t *)(r_out + n_out), *r_nf = r_milli + n_out;
  if ((rc = hg_search_merge(c0, (uint32_t)parts, g_hits, g_found, b.data(), n_qry, top_k, r_out, r_nf, ani_milli ? r_milli : nullptr)))
    return rc;
  HG_CUDA(cudaMemcpyAsync(out, r_out, n_out * sizeof(hg_hit), cudaMemcpyDeviceToHost, c0->stream));
  HG_CUDA(cudaMemcpyAsync(n_found, r_nf, (size_t)n_qry * 4, cudaMemcpyDeviceToHost, c0->stream));
  if (ani_milli) HG_CUDA(cudaMemcpyAsync(ani_milli, r_milli, n_out * 4, cudaMemcpyDeviceToHost, c0->stream));
  HG_CUDA(cudaStreamSynchronize(c0->stream));
  return HG_OK;
}

// hg_cluster_packed over all GPUs of the group (DESIGN.md §4.9).  The upper triangle is cut by query column into one range
// per member, b_k = n sqrt(k / parts) rounded to 256, which gives every member about the same number of pairs: member m
// takes the columns [b_m, b_m+1) against the refs [0, b_m+1).  It copies packed rows [0, b_m+1) over its own PCIe link,
// unpacks and prepares them, and builds its own forest of those rows with the single-GPU windows and hooks.  As many
// members as give each at least 2^23 pairs (a 4096-row triangle) take part.  One host thread per GPU drives its members:
// members that share a device ordinal run one after another (as in hg_group_search_packed).  The forests are copied to
// GPU 0 and united there into iota(n): the partition of a union of edge sets is the union-find over the members' forests,
// so the result is the single-GPU one.  The only exchange is one label per row and member, so no windows.
extern "C" int hg_group_cluster_packed(hg_group *g, const uint8_t *packed, uint64_t stride, const uint8_t *quant_bits, const int32_t *norm2,
                                       uint32_t n, uint32_t hv_d, uint32_t ksize, float ani_th, int path, uint32_t *rep,
                                       uint32_t *n_clusters) {
  if (!g) { hg_set_error("hg_group_cluster_packed: NULL argument"); return HG_E_INVALID; }
  for (int k = 0; k < g->n; ++k) hg_cluster_stats_reset(g->ctx[k]);  // a member without columns reports no run
  hg_packed_rows R = {packed, stride, quant_bits, norm2, n};
  const char *who = "hg_group_cluster_packed";
  int rc;
  if ((rc = hg_packed_args_check(who, R, R, hv_d)) || (rc = hg_cluster_check(who, n, rep, hv_d, ani_th, path))) return rc;
  const uint64_t pairs = n ? (uint64_t)n * (n - 1) / 2 : 0;
  const int parts = (int)std::min<uint64_t>((uint64_t)g->n, std::max<uint64_t>(1, pairs >> 23));
  if (parts == 1) return hg_cluster_packed_host(g->ctx[0], who, R, hv_d, ksize, ani_th, path, rep, n_clusters);
  bool same;
  hg_packed_rows Q = R;
  if ((rc = hg_packed_rows_check(who, &R, &Q, hv_d, &same))) return rc;
  std::vector<uint32_t> b(parts + 1, n);
  b[0] = 0;
  for (int k = 1; k < parts; ++k) {
    const uint32_t want = (uint32_t)(std::lround((double)n * std::sqrt((double)k / parts) / 256.0) * 256);
    b[k] = std::min(n, std::max(b[k - 1], want));
  }
  std::vector<uint32_t *> d_rep(parts);
  std::vector<int> rcs(parts, HG_OK);
  std::vector<std::string> msgs(parts);
  auto member = [&](int m) -> int {
    hg_ctx *c = g->ctx[m];
    HG_CUDA(cudaSetDevice(c->device));
    return hg_cluster_packed_run(c, R.rows(0, b[m + 1]), b[m], hv_d, ksize, ani_th, path, &d_rep[m], nullptr, nullptr);
  };
  std::vector<std::thread> th;
  for (int k = 0; k < parts; ++k) {
    bool first_on_device = true;
    for (int l = 0; l < k; ++l) first_on_device &= g->ctx[l]->device != g->ctx[k]->device;
    if (!first_on_device) continue;
    th.emplace_back([&, k]() {
      for (int m = k; m < parts; ++m) {
        if (g->ctx[m]->device != g->ctx[k]->device) continue;
        if ((rcs[m] = member(m))) msgs[m] = hg_last_error();
      }
    });
  }
  for (auto &t : th) t.join();
  for (int k = 0; k < parts; ++k)
    if (rcs[k]) { hg_set_error("GPU %d (columns %u..%u): %s", g->ctx[k]->device, b[k], b[k + 1], msgs[k].c_str()); return rcs[k]; }
  // merge on GPU 0: iota(n), then every member's forest gathered next to it and united into it
  hg_ctx *c0 = g->ctx[0];
  HG_CUDA(cudaSetDevice(c0->device));
  uint64_t words = n;
  for (int k = 0; k < parts; ++k) words += b[k + 1];
  void *d_buf;
  if ((rc = hg_scratch(c0, HG_S_SORT_TMP, words * 4, &d_buf))) return rc;
  uint32_t *merged = (uint32_t *)d_buf, *f = merged + n;
  if ((rc = hg_launch_cluster_iota(c0, merged, n))) return rc;
  for (int k = 0; k < parts; ++k) {
    if (b[k + 1]) HG_CUDA(cudaMemcpyPeerAsync(f, c0->device, d_rep[k], g->ctx[k]->device, (size_t)b[k + 1] * 4, c0->stream));
    if ((rc = hg_launch_cluster_hook_labels(c0, merged, f, b[k + 1]))) return rc;
    f += b[k + 1];
  }
  return hg_cluster_finish(c0, merged, n, rep, n_clusters);
}

// hg_ani_matrix_packed over all GPUs of the group (DESIGN.md §4.11).  The ref rows are cut into one contiguous range per
// member with about the same number of output entries: b_k = n sqrt(k / parts) in lower mode, n_ref k / parts for a
// rectangle.  Member m copies the packed rows it reads over its own PCIe link (lower: rows [0, b_m+1); rectangle: its
// range and every query row), computes its bands and copies them straight into its part of `out`, which is page-locked
// once for all members.  As many members as give each at least 2^23 entries take part (cluster's rule).  One host thread
// per GPU drives its members; members that share a device ordinal run one after another.  Every cell is the exact value
// whatever the kernel, so the result is byte-identical to hg_ani_matrix_packed.
extern "C" int hg_group_ani_matrix_packed(hg_group *g, const uint8_t *ref_packed, uint64_t ref_stride, const uint8_t *ref_bits,
                                          const int32_t *ref_norm2, uint32_t n_ref, const uint8_t *qry_packed, uint64_t qry_stride,
                                          const uint8_t *qry_bits, const int32_t *qry_norm2, uint32_t n_qry, uint32_t hv_d,
                                          uint32_t ksize, int path, int lower, float *out, uint64_t ld) {
  const char *who = "hg_group_ani_matrix_packed";
  if (!g) { hg_set_error("%s: NULL argument", who); return HG_E_INVALID; }
  hg_packed_rows R = {ref_packed, ref_stride, ref_bits, ref_norm2, n_ref}, Q = {qry_packed, qry_stride, qry_bits, qry_norm2, n_qry};
  const bool same = R.packed == Q.packed && R.bits == Q.bits && R.norm == Q.norm && R.n == Q.n;
  int rc;
  if ((rc = hg_packed_args_check(who, R, Q, hv_d)) || (rc = hg_matrix_check(who, same, n_ref, n_qry, hv_d, path, lower, out, ld))) return rc;
  const uint64_t entries = hg_matrix_entries(n_ref, n_qry, lower);
  const int parts = (int)std::min<uint64_t>((uint64_t)g->n, std::max<uint64_t>(1, entries >> 23));
  if (parts == 1)
    return hg_ani_matrix_packed(g->ctx[0], ref_packed, ref_stride, ref_bits, ref_norm2, n_ref, qry_packed, qry_stride, qry_bits, qry_norm2,
                                n_qry, hv_d, ksize, path, lower, out, ld);
  bool same2;
  if ((rc = hg_packed_rows_check(who, &R, &Q, hv_d, &same2))) return rc;
  std::vector<uint32_t> b(parts + 1, n_ref);
  b[0] = 0;
  for (int k = 1; k < parts; ++k) {
    const uint32_t want = lower ? (uint32_t)std::lround((double)n_ref * std::sqrt((double)k / parts))
                                : (uint32_t)((uint64_t)n_ref * k / parts);
    b[k] = std::min(n_ref, std::max(b[k - 1], want));
  }
  HostPin pin;
  HG_CUDA(cudaSetDevice(g->ctx[0]->device));
  if ((rc = pin.pin(out, (lower ? entries : (uint64_t)(n_ref - 1) * ld + n_qry) * 4))) return rc;
  std::vector<int> rcs(parts, HG_OK);
  std::vector<std::string> msgs(parts);
  auto member = [&](int m) -> int {
    hg_ctx *c = g->ctx[m];
    if (b[m] == b[m + 1]) return HG_OK;
    if (lower)
      return hg_matrix_packed_run(c, R.rows(0, b[m + 1]), R.rows(0, b[m + 1]), true, hv_d, ksize, path, true, b[m],
                                  out + (uint64_t)b[m] * ((uint64_t)b[m] - 1) / 2, ld);
    return hg_matrix_packed_run(c, R.rows(b[m], b[m + 1] - b[m]), Q, false, hv_d, ksize, path, false, 0, out + (uint64_t)b[m] * ld, ld);
  };
  for (int k = 0; k < g->n; ++k) {  // a member without rows reports no run
    memset(g->ctx[k]->matrix_stats, 0, sizeof(g->ctx[k]->matrix_stats));
    for (float &t : g->ctx[k]->matrix_ms) t = -1.0f;
  }
  std::vector<std::thread> th;
  for (int k = 0; k < parts; ++k) {
    bool first_on_device = true;
    for (int l = 0; l < k; ++l) first_on_device &= g->ctx[l]->device != g->ctx[k]->device;
    if (!first_on_device) continue;
    th.emplace_back([&, k]() {
      for (int m = k; m < parts; ++m) {
        if (g->ctx[m]->device != g->ctx[k]->device) continue;
        if ((rcs[m] = member(m))) msgs[m] = hg_last_error();
      }
    });
  }
  for (auto &t : th) t.join();
  for (int k = 0; k < parts; ++k)
    if (rcs[k]) { hg_set_error("GPU %d (rows %u..%u): %s", g->ctx[k]->device, b[k], b[k + 1], msgs[k].c_str()); return rcs[k]; }
  return HG_OK;
}
