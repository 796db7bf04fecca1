// Multi-GPU layer of libgbm_b200.so (include/gbm_b200.h, section "multi-GPU"): marker shards over the GPUs of one
// box, NCCL inside the library.
//
// The reference's parallel axis is the marker loop (`Threads.@threads for j = 1:l`, /root/reference/src/gwas.jl:239,
// :363).  Here every GPU owns a contiguous column block; the pieces of gwasprep / gwasols / gwaslmm need
//   GRM (gwas.jl:120, :124)            one all-reduce of the n x n partial sums (+ one scalar)
//   K standardisation + PC1 (:130,:234) columns of K sharded; all-reduce of the row sums, then of one n-vector per
//                                       Lanczos step
//   filter (:113)                       local; idx_cols concatenated in shard order with the prefix of the counts
//   marker loop (:239-249, :363-389)    nothing; results gathered in locus order
// A group is either this process driving all its GPUs (one host thread + one State per GPU, ncclCommInitAll) or
// one process per GPU (ncclCommInitRank on the gbm_init device).  The per-GPU work is done through the library's
// own single-GPU entry points, each running on the State bound to the calling thread.
#include "../../include/gbm_b200.h"

#include <dlfcn.h>
#include <nccl.h>
#include <string.h>

#include <algorithm>
#include <array>
#include <chrono>
#include <condition_variable>
#include <functional>
#include <memory>
#include <mutex>
#include <thread>
#include <vector>

#include "common.cuh"
#include "kernels.h"

using namespace gbm;

// NCCL is bound at run time, at the first group creation: a process that already holds a libnccl.so.2 (PyTorch
// ships and loads its own, newer than the system's) must keep using THAT copy -- a second library with the same
// soname cannot be loaded next to it, and loading the system's first would break a later `import torch`.  Order:
// an already loaded libnccl.so.2, then $GBM_NCCL_LIB, then the system's libnccl.so.2.
namespace {
struct NcclApi {
  decltype(&ncclGetErrorString) GetErrorString = nullptr;
  decltype(&ncclCommInitAll) CommInitAll = nullptr;
  decltype(&ncclGetUniqueId) GetUniqueId = nullptr;
  decltype(&ncclCommInitRank) CommInitRank = nullptr;
  decltype(&ncclCommDestroy) CommDestroy = nullptr;
  decltype(&ncclAllReduce) AllReduce = nullptr;
  decltype(&ncclAllGather) AllGather = nullptr;
  decltype(&ncclBroadcast) Broadcast = nullptr;
  decltype(&ncclGroupStart) GroupStart = nullptr;
  decltype(&ncclGroupEnd) GroupEnd = nullptr;
};

const NcclApi& nccl() {
  static std::mutex m;
  static NcclApi api;
  static bool ready = false;
  std::lock_guard<std::mutex> lk(m);
  if (ready) return api;
  void* h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_NOLOAD);
  if (!h)
    if (const char* e = getenv("GBM_NCCL_LIB")) h = dlopen(e, RTLD_NOW | RTLD_GLOBAL);
  if (!h) h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
  if (!h) throw Error{GBM_ERR_CUDA, std::string("multi-GPU groups need NCCL: libnccl.so.2 could not be loaded (") + dlerror() + ")"};
  auto sym = [&](const char* name) {
    void* p = dlsym(h, name);
    if (!p) throw Error{GBM_ERR_CUDA, std::string("libnccl.so.2 lacks ") + name};
    return p;
  };
  api.GetErrorString = reinterpret_cast<decltype(api.GetErrorString)>(sym("ncclGetErrorString"));
  api.CommInitAll = reinterpret_cast<decltype(api.CommInitAll)>(sym("ncclCommInitAll"));
  api.GetUniqueId = reinterpret_cast<decltype(api.GetUniqueId)>(sym("ncclGetUniqueId"));
  api.CommInitRank = reinterpret_cast<decltype(api.CommInitRank)>(sym("ncclCommInitRank"));
  api.CommDestroy = reinterpret_cast<decltype(api.CommDestroy)>(sym("ncclCommDestroy"));
  api.AllReduce = reinterpret_cast<decltype(api.AllReduce)>(sym("ncclAllReduce"));
  api.AllGather = reinterpret_cast<decltype(api.AllGather)>(sym("ncclAllGather"));
  api.Broadcast = reinterpret_cast<decltype(api.Broadcast)>(sym("ncclBroadcast"));
  api.GroupStart = reinterpret_cast<decltype(api.GroupStart)>(sym("ncclGroupStart"));
  api.GroupEnd = reinterpret_cast<decltype(api.GroupEnd)>(sym("ncclGroupEnd"));
  ready = true;
  return api;
}
}  // namespace

#define GBM_NCCL(call)                                                                                            \
  do {                                                                                                            \
    ncclResult_t r__ = (call);                                                                                    \
    if (r__ != ncclSuccess)                                                                                       \
      throw ::gbm::Error{GBM_ERR_CUDA, std::string(#call) + ": " + nccl().GetErrorString(r__) + " (" + __FILE__ + ":" + \
                                           std::to_string(__LINE__) + ")"};                                       \
  } while (0)

namespace {

double now_ms() {
  return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count();
}
int64_t round_up(int64_t x, int64_t m) { return (x + m - 1) / m * m; }

// result of a single-GPU entry point called on the current thread's State
void ok(int rc) {
  if (rc != GBM_OK) throw Error{rc, std::string(gbm_last_error())};
}

// stream-ordered device scratch on the calling thread's State
template <typename T>
struct Dev {
  T* p = nullptr;
  cudaStream_t s;
  explicit Dev(size_t count) : s(state().stream) {
    if (count) GBM_CUDA(cudaMallocAsync(reinterpret_cast<void**>(&p), count * sizeof(T), s));
  }
  ~Dev() {
    if (p) cudaFreeAsync(p, s);
  }
  Dev(const Dev&) = delete;
  Dev& operator=(const Dev&) = delete;
};

__global__ void add_offset_kernel(int64_t* __restrict__ v, int64_t count, int64_t off) {
  const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i < count) v[i] += off;
}

// one persistent host thread per GPU of a local group
struct Worker {
  std::thread th;
  std::mutex m;
  std::condition_variable cv;
  std::function<void()> job;
  bool busy = false, quit = false;
  int rc = GBM_OK;
  std::string err;

  void start(State* st) {
    th = std::thread([this, st] {
      bind_state(st);
      std::unique_lock<std::mutex> lk(m);
      for (;;) {
        cv.wait(lk, [this] { return busy || quit; });
        if (quit) return;
        lk.unlock();
        int r = GBM_OK;
        std::string e;
        try {
          job();
        } catch (const Error& x) {
          r = x.code;
          e = x.msg;
        } catch (const std::exception& x) {
          r = GBM_ERR_RUNTIME;
          e = std::string("internal: ") + x.what();
        }
        lk.lock();
        rc = r;
        err = e;
        busy = false;
        cv.notify_all();
      }
    });
  }
  void post(std::function<void()> f) {
    std::lock_guard<std::mutex> lk(m);
    job = std::move(f);
    busy = true;
    cv.notify_all();
  }
  void wait() {
    std::unique_lock<std::mutex> lk(m);
    cv.wait(lk, [this] { return !busy; });
  }
  void stop() {
    {
      std::lock_guard<std::mutex> lk(m);
      quit = true;
      cv.notify_all();
    }
    if (th.joinable()) th.join();
  }
};

}  // namespace

// one GPU's side of the peer-memory all-reduce of the sharded Lanczos step (lanczos.cu: peer_sum_kernel)
struct PeerState {
  PeerMailbox mb;
  double* slots = nullptr;               // this GPU's mailbox: 2 x W x npad entries of 16 bytes (cudaMalloc: shareable by CUDA IPC)
  std::vector<void*> opened;             // CUDA IPC mappings of the peers' mailboxes (rank groups)
  unsigned long long step = 0;
};

struct gbm_group {
  std::vector<PeerState> peer;           // per local GPU
  int64_t peer_npad = 0;                 // 0: no mailboxes yet; -1: peer access not available (NCCL is used)
  int world = 1, n_local = 1, first_rank = 0;
  bool threaded = false;  // local group: a worker thread per GPU; rank group: inline on the caller's thread
  std::vector<std::unique_ptr<State>> owned;
  std::vector<State*> ctx;
  std::vector<ncclComm_t> comm;
  std::vector<std::unique_ptr<Worker>> workers;
  std::mutex mutex;  // group entry points are serialised

  // f(g) on the State of every local GPU; the first failure (lowest g) is re-thrown on the calling thread after
  // ALL of them have returned
  template <typename F>
  void run(F f) {
    if (!threaded) {
      State* prev = &state();
      bind_state(ctx[0]);
      try {
        GBM_CUDA(cudaSetDevice(ctx[0]->device));
        f(0);
      } catch (...) {
        bind_state(prev == ctx[0] ? nullptr : prev);
        throw;
      }
      bind_state(prev == ctx[0] ? nullptr : prev);
      return;
    }
    for (int g = 0; g < n_local; ++g) workers[g]->post([f, g] { f(g); });
    for (int g = 0; g < n_local; ++g) workers[g]->wait();
    for (int g = 0; g < n_local; ++g)
      if (workers[g]->rc != GBM_OK) throw Error{workers[g]->rc, "GPU " + std::to_string(ctx[g]->device) + ": " + workers[g]->err};
  }

  // A phase of rank-local work that is followed by a collective: when it fails on some process only, the others
  // must not walk into the collective and hang there.  Local groups are covered by run() (every thread returns
  // before anything is re-thrown); rank groups agree on a status word first.
  template <typename F>
  void phase(F f) {
    if (threaded || world == 1) {
      run(f);
      return;
    }
    int rc = GBM_OK;
    std::string msg;
    try {
      run(f);
    } catch (const Error& e) {
      rc = e.code;
      msg = e.msg;
    }
    int worst = rc;
    run([&](int) {
      Dev<int> d(1);
      cudaStream_t s = state().stream;
      GBM_CUDA(cudaMemcpyAsync(d.p, &rc, sizeof(int), cudaMemcpyHostToDevice, s));
      GBM_NCCL(nccl().AllReduce(d.p, d.p, 1, ncclInt, ncclMax, comm[0], s));
      GBM_CUDA(cudaMemcpyAsync(&worst, d.p, sizeof(int), cudaMemcpyDeviceToHost, s));
      GBM_CUDA(cudaStreamSynchronize(s));
    });
    if (rc != GBM_OK) throw Error{rc, msg};
    if (worst != GBM_OK) throw Error{worst, "another rank of the group failed in this call (see its error message)"};
  }

  int rank_of(int g) const { return first_rank + g; }

  // sum / min / max of `count` doubles per local GPU over all ranks; vals[g] is overwritten with the result
  void reduce_host(std::vector<std::vector<double>>& vals, ncclRedOp_t op) {
    const size_t count = vals[0].size();
    if (world == n_local) {  // every rank is here: combine on the host, fixed order
      std::vector<double> acc = vals[0];
      for (int g = 1; g < n_local; ++g)
        for (size_t i = 0; i < count; ++i)
          acc[i] = op == ncclSum ? acc[i] + vals[g][i] : op == ncclMin ? std::min(acc[i], vals[g][i]) : std::max(acc[i], vals[g][i]);
      for (auto& v : vals) v = acc;
      return;
    }
    run([&](int g) {
      Dev<double> d(count);
      cudaStream_t s = state().stream;
      GBM_CUDA(cudaMemcpyAsync(d.p, vals[g].data(), sizeof(double) * count, cudaMemcpyHostToDevice, s));
      GBM_NCCL(nccl().AllReduce(d.p, d.p, count, ncclDouble, op, comm[g], s));
      GBM_CUDA(cudaMemcpyAsync(vals[g].data(), d.p, sizeof(double) * count, cudaMemcpyDeviceToHost, s));
      GBM_CUDA(cudaStreamSynchronize(s));
    });
  }

  // per-rank counts (world entries) from the local ones
  std::vector<int64_t> all_counts(const std::vector<int64_t>& local) {
    std::vector<int64_t> all(world, 0);
    if (world == n_local) {
      for (int g = 0; g < n_local; ++g) all[g] = local[g];
      return all;
    }
    run([&](int g) {
      Dev<int64_t> d(world);
      cudaStream_t s = state().stream;
      GBM_CUDA(cudaMemcpyAsync(d.p + rank_of(g), &local[g], sizeof(int64_t), cudaMemcpyHostToDevice, s));
      GBM_NCCL(nccl().AllGather(d.p + rank_of(g), d.p, 1, ncclInt64, comm[g], s));
      GBM_CUDA(cudaMemcpyAsync(all.data(), d.p, sizeof(int64_t) * world, cudaMemcpyDeviceToHost, s));
      GBM_CUDA(cudaStreamSynchronize(s));
    });
    return all;
  }
};

namespace {

// Must run inside group.run: gathers, on the calling thread's GPU g, `height` rows of per-marker values from every
// rank into `host` (full length, locus order; row pitch `total` elements).  src: this GPU's block, `counts[rank]`
// elements per row, rows `counts[rank]` apart.  offs = exclusive prefix of counts.
template <typename T>
void gather_rows(gbm_group& G, int g, const T* src, const std::vector<int64_t>& counts, const std::vector<int64_t>& offs,
                 int64_t total, int64_t height, T* host) {
  if (!host || height <= 0) return;
  cudaStream_t s = state().stream;
  const int me = G.rank_of(g);
  if (G.world == G.n_local) {  // every block is in this process: straight to its slice of the caller's array
    if (counts[me] > 0)
      GBM_CUDA(cudaMemcpy2DAsync(host + offs[me], total * sizeof(T), src, counts[me] * sizeof(T), counts[me] * sizeof(T),
                                 height, cudaMemcpyDeviceToHost, s));
    return;
  }
  // one process per GPU: blocks travel over NVLink into a rank-major device buffer, then to the host array
  Dev<T> full(static_cast<size_t>(total) * height);
  GBM_NCCL(nccl().GroupStart());
  for (int r = 0; r < G.world; ++r) {
    const size_t bytes = static_cast<size_t>(counts[r]) * height * sizeof(T);
    if (!bytes) continue;
    T* slot = full.p + offs[r] * height;
    GBM_NCCL(nccl().Broadcast(r == me ? static_cast<const void*>(src) : static_cast<const void*>(slot), slot, bytes, ncclUint8,
                           r, G.comm[g], s));
  }
  GBM_NCCL(nccl().GroupEnd());
  for (int r = 0; r < G.world; ++r)
    if (counts[r] > 0)
      GBM_CUDA(cudaMemcpy2DAsync(host + offs[r], total * sizeof(T), full.p + offs[r] * height, counts[r] * sizeof(T),
                                 counts[r] * sizeof(T), height, cudaMemcpyDeviceToHost, s));
  GBM_CUDA(cudaStreamSynchronize(s));  // `full` is released when this returns
}

std::vector<int64_t> prefix(const std::vector<int64_t>& c) {
  std::vector<int64_t> o(c.size(), 0);
  for (size_t i = 1; i < c.size(); ++i) o[i] = o[i - 1] + c[i - 1];
  return o;
}

struct NcclSum : ShardedAllReduce {
  ncclComm_t comm;
  cudaStream_t s;
  NcclSum(ncclComm_t c, cudaStream_t st) : comm(c), s(st) {}
  void sum(double* buf, int64_t count) override {
    GBM_NCCL(nccl().AllReduce(buf, buf, static_cast<size_t>(count), ncclDouble, ncclSum, comm, s));
  }
};

struct PeerSum : NcclSum {  // the per-step all-reduce over peer memory, fused with the partial-sum reduction
  PeerState* ps;
  PeerSum(ncclComm_t c, cudaStream_t st, PeerState* p) : NcclSum(c, st), ps(p) {}
  void sum_partials(const double* partial, int chunks, int64_t n, double* out, cudaStream_t stream) override {
    launch_peer_sum(ps->mb, partial, chunks, n, ++ps->step, out, stream);
  }
};

void free_peer(gbm_group& G) {
  if (G.peer.empty()) return;
  try {
    G.run([&](int g) {
      PeerState& ps = G.peer[g];
      cudaStreamSynchronize(state().stream);
      for (void* p : ps.opened) cudaIpcCloseMemHandle(p);
      ps.opened.clear();
      if (ps.slots) cudaFree(ps.slots);
      if (ps.mb.error) cudaFree(ps.mb.error);
      ps = PeerState();
    });
  } catch (...) {
  }
  G.peer.clear();
  G.peer_npad = 0;
}

// Mailboxes for n-vectors on every GPU of the group, visible to every other GPU: peer access inside one process,
// CUDA IPC mappings between processes.  Returns false (and remembers it) when the GPUs cannot reach each other's
// memory -- the Lanczos step then uses NCCL.  The mailboxes are sized ONCE, for the largest n the fused Lanczos step
// takes (kLanczosFusedMaxN: 3 MB per GPU at 8 ranks), and live as long as the group: a mailbox is never freed while
// another process may still map it.
bool ensure_peer(gbm_group& G, int64_t n) {
  const char* env = getenv("GBM_PC1_PEER");  // read per call: the tests compare both routes in one process
  if ((env && atoi(env) == 0) || G.world > PeerMailbox::kMaxRanks || G.world < 2 || G.peer_npad < 0) return false;
  if (n > kLanczosFusedMaxN) return false;  // larger n take the two-pass step, whose all-reduce is NCCL's
  const int64_t npad = round_up(kLanczosFusedMaxN, 256);
  if (G.peer_npad == npad) return true;
  G.peer.assign(G.n_local, PeerState());
  const int W = G.world;
  std::vector<int> okv(G.n_local, 1);
  // (1) allocate, and in a local group switch peer access on
  G.phase([&](int g) {
    PeerState& ps = G.peer[g];
    if (G.threaded) {
      for (int h = 0; h < G.n_local; ++h) {
        if (h == g) continue;
        int can = 0;
        GBM_CUDA(cudaDeviceCanAccessPeer(&can, G.ctx[g]->device, G.ctx[h]->device));
        if (!can) {
          okv[g] = 0;
          return;
        }
        cudaError_t e = cudaDeviceEnablePeerAccess(G.ctx[h]->device, 0);
        if (e == cudaErrorPeerAccessAlreadyEnabled) cudaGetLastError();
        else GBM_CUDA(e);
      }
    }
    GBM_CUDA(cudaMalloc(reinterpret_cast<void**>(&ps.slots), sizeof(double) * 2 * 2 * W * npad));
    GBM_CUDA(cudaMalloc(reinterpret_cast<void**>(&ps.mb.error), sizeof(int)));
    GBM_CUDA(cudaMemset(ps.slots, 0, sizeof(double) * 2 * 2 * W * npad));  // stamp 0: no step has it
    GBM_CUDA(cudaMemset(ps.mb.error, 0, sizeof(int)));
    GBM_CUDA(cudaDeviceSynchronize());
  });
  std::vector<std::vector<double>> okr(G.n_local, std::vector<double>(1, 1.0));
  for (int g = 0; g < G.n_local; ++g) okr[g][0] = okv[g];
  // (2) every rank learns every mailbox address
  try {
    if (G.threaded) {
      G.reduce_host(okr, ncclMin);
      if (okr[0][0] < 0.5) throw Error{GBM_ERR_RUNTIME, "no peer access"};
      for (int g = 0; g < G.n_local; ++g)
        for (int q = 0; q < W; ++q) G.peer[g].mb.slots[q] = G.peer[q].slots;
    } else {
      // one process per GPU: CUDA IPC handles travel through an all-gather, every peer mailbox is mapped here.  The
      // mapping can fail on some ranks only (a peer on another node, no P2P path): G.phase makes that a common verdict.
      struct Handles {
        cudaIpcMemHandle_t slots;
      };
      static_assert(sizeof(Handles) == 64, "a 64-byte IPC handle");
      std::vector<Handles> all(W);
      G.run([&](int g) {
        PeerState& ps = G.peer[g];
        cudaStream_t st = state().stream;
        const int me = G.rank_of(g);
        GBM_CUDA(cudaIpcGetMemHandle(&all[me].slots, ps.slots));
        Dev<uint8_t> d(sizeof(Handles) * W);
        GBM_CUDA(cudaMemcpyAsync(d.p + sizeof(Handles) * me, &all[me], sizeof(Handles), cudaMemcpyHostToDevice, st));
        GBM_NCCL(nccl().AllGather(d.p + sizeof(Handles) * me, d.p, sizeof(Handles), ncclUint8, G.comm[g], st));
        GBM_CUDA(cudaMemcpyAsync(all.data(), d.p, sizeof(Handles) * W, cudaMemcpyDeviceToHost, st));
        GBM_CUDA(cudaStreamSynchronize(st));
      });
      G.phase([&](int g) {
        PeerState& ps = G.peer[g];
        const int me = G.rank_of(g);
        for (int q = 0; q < W; ++q) {
          if (q == me) {
            ps.mb.slots[q] = ps.slots;
            continue;
          }
          void* ps_q = nullptr;
          GBM_CUDA(cudaIpcOpenMemHandle(&ps_q, all[q].slots, cudaIpcMemLazyEnablePeerAccess));
          ps.opened.push_back(ps_q);
          ps.mb.slots[q] = static_cast<double*>(ps_q);
        }
      });
    }
  } catch (const Error&) {
    // Falling back is the SAME decision on every rank: one process decides for a local group, G.phase agreed on the
    // failure for a rank group.  The Lanczos step then uses NCCL.
    cudaGetLastError();
    free_peer(G);
    G.peer_npad = -1;
    return false;
  }
  for (int g = 0; g < G.n_local; ++g) {
    G.peer[g].mb.world = W;
    G.peer[g].mb.me = G.rank_of(g);
    G.peer[g].mb.mine = G.peer[g].mb.slots[G.rank_of(g)];
    G.peer[g].mb.npad = npad;
  }
  G.peer_npad = npad;
  return true;
}

}  // namespace

struct gbm_sharded {
  gbm_group* grp = nullptr;
  int64_t n = 0, p = 0;
  std::vector<gbm_matrix*> local;  // one block per local GPU
  bool owned = true;
  int packed = 0;
  std::vector<int64_t> ncols, col0;  // per rank of the group
  std::vector<double*> dK;           // per local GPU: the GRM left resident by gbm_sharded_grm (n x n)
  bool have_K = false;
};

namespace {

void check_group(const gbm_group* g) {
  if (!g) GBM_THROW(GBM_ERR_ARGUMENT, "null group handle");
}
void check_sharded(const gbm_sharded* m) {
  if (!m || !m->grp) GBM_THROW(GBM_ERR_ARGUMENT, "null sharded-matrix handle");
}

void free_blocks(gbm_sharded* m) {
  gbm_group& G = *m->grp;
  G.run([&](int g) {
    if (m->owned && m->local[g]) gbm_matrix_free(m->local[g]);
    m->local[g] = nullptr;
    if (m->dK[g]) {
      cudaStreamSynchronize(state().stream);
      cudaFree(m->dK[g]);
      m->dK[g] = nullptr;
    }
  });
}

// column ranges of every rank from the local block widths
void finish_layout(gbm_sharded* m) {
  gbm_group& G = *m->grp;
  std::vector<int64_t> loc(G.n_local);
  for (int g = 0; g < G.n_local; ++g) ok(gbm_matrix_info(m->local[g], nullptr, &loc[g], nullptr, nullptr));
  m->ncols = G.all_counts(loc);
  m->col0 = prefix(m->ncols);
  m->p = m->col0.back() + m->ncols.back();
}

void ensure_dK(gbm_sharded* m, int g) {
  if (!m->dK[g]) {
    cudaError_t e = cudaMalloc(reinterpret_cast<void**>(&m->dK[g]), sizeof(double) * m->n * m->n);
    if (e != cudaSuccess) GBM_THROW(GBM_ERR_CUDA, std::string("cudaMalloc of the GRM failed: ") + cudaGetErrorString(e));
  }
}

struct GrmTimes {
  double grm_ms = 0, allreduce_ms = 0;
};

// per-GPU partials -> all-reduce -> scale + mirror; the GRM stays resident in m->dK on every GPU
GrmTimes sharded_grm(gbm_sharded* m, int grm_type, int ploidy, int flags, int64_t* launches) {
  gbm_group& G = *m->grp;
  if (grm_type != GBM_GRM_SIMPLE && grm_type != GBM_GRM_PLOIDY_AWARE)
    GBM_THROW(GBM_ERR_ARGUMENT, "Unrecognised `GRM_type`. Please select from:\n\t‣ simple\n\t‣ ploidy-aware");
  if (grm_type == GBM_GRM_PLOIDY_AWARE && ploidy < 1) GBM_THROW(GBM_ERR_ARGUMENT, "gbm_grm: ploidy must be >= 1");
  const bool pa = grm_type == GBM_GRM_PLOIDY_AWARE;
  const int centre = pa ? 1 : ((flags & GBM_GRM_NO_CENTRE) ? 0 : 1);
  const int64_t n = m->n;
  std::vector<std::vector<double>> sumq(G.n_local, std::vector<double>(1, 0.0));
  GrmTimes t;
  m->have_K = false;
  const double t0 = now_ms();
  G.phase([&](int g) {
    ensure_dK(m, g);
    GBM_CUDA(cudaMemsetAsync(m->dK[g], 0, sizeof(double) * n * n, state().stream));  // same stream as the contraction
    double s = 0.0;
    ok(gbm_grm_accumulate(m->local[g], centre, m->dK[g], pa ? &s : nullptr, nullptr));
    sumq[g][0] = s;
    if (launches) launches[g] += state().launches;
  });
  const double t1 = now_ms();
  if (pa) G.reduce_host(sumq, ncclSum);
  double scale = 1.0 / static_cast<double>(m->p);
  if (pa) {
    if (!(sumq[0][0] > 0.0)) GBM_THROW(GBM_ERR_RUNTIME, "gbm_grm: sum q(1-q) is not positive (all loci fixed)");
    scale = static_cast<double>(ploidy) / sumq[0][0];
  }
  G.run([&](int g) {
    cudaStream_t s = state().stream;
    if (G.world > 1)
      GBM_NCCL(nccl().AllReduce(m->dK[g], m->dK[g], static_cast<size_t>(n) * n, ncclDouble, ncclSum, G.comm[g], s));
    ok(gbm_grm_finalize(m->dK[g], n, scale));  // synchronises the stream
    if (launches) launches[g] += 1;
  });
  t.grm_ms = t1 - t0;
  t.allreduce_ms = now_ms() - t1;
  m->have_K = true;
  return t;
}

// K standardisation + PC1 from the GRM resident in m->dK (every GPU holds all of it).  Returns eig_ms.
// pc1_host (n) is filled on this process; steps (nullable) gets the Lanczos step count.
double sharded_kstd_pc1(gbm_sharded* m, double* pc1_host, int* steps, int64_t* launches) {
  gbm_group& G = *m->grp;
  const int64_t n = m->n;
  if (!m->have_K) GBM_THROW(GBM_ERR_ARGUMENT, "gbm_sharded_kstd_pc1: no resident GRM (call gbm_sharded_grm first or pass K)");
  static const bool no_shard = [] { const char* e = getenv("GBM_PC1_SHARDED"); return e && atoi(e) == 0; }();
  std::vector<double> eig(G.n_local, 0.0);
  std::vector<int> conv(G.n_local, 0), iters(G.n_local, 0);
  // below n ~ 4,000 a step's two passes over the block cost less than the all-reduce that sharding adds
  const bool sharded = G.world > 1 && n >= 4096 && !no_shard;
  if (sharded) {
    const int64_t ld = round_up(n, 16);
    // the per-step all-reduce: one kernel over peer memory (NVLink stores into every GPU's mailbox) when the GPUs can
    // reach each other's memory, NCCL otherwise
    const bool peer = ensure_peer(G, n);
    G.run([&](int g) {
      State& st = state();
      cudaStream_t s = st.stream;
      const int r = G.rank_of(g);
      const int64_t c0 = n * r / G.world, c1 = n * (r + 1) / G.world, nc = c1 - c0;
      // this rank's column block of K, padded to the TMA pitch
      Dev<double> Z(static_cast<size_t>(ld) * nc), rec(static_cast<size_t>(nc) * scan_record_stride(0, true)), mean(nc), sd(nc),
          rowsum(round_up(n, 2)), x(n);
      if (ld != n) GBM_CUDA(cudaMemsetAsync(Z.p, 0, sizeof(double) * ld * nc, s));
      GBM_CUDA(cudaMemcpy2DAsync(Z.p, ld * sizeof(double), m->dK[g] + c0 * n, n * sizeof(double), n * sizeof(double), nc,
                                 cudaMemcpyDeviceToDevice, s));
      // K = (K .- mean(K, dims=1)) ./ std(K, dims=1)   (gwas.jl:130): column statistics are local to the block
      launch_scan_sums(Z.p, n, nc, ld, nullptr, 0, 0, true, rec.p, st.sm_count, s);
      launch_colstats_finalize(rec.p, scan_record_stride(0, true), n, nc, mean.p, sd.p, nullptr, nullptr, s);
      launch_k_standardise(Z.p, n, nc, ld, mean.p, sd.p, s);
      // PCA centres the rows (gwas.jl:234): row sums of the block, summed over the ranks
      block_row_sums(Z.p, n, nc, ld, rowsum.p, s);
      NcclSum nccl_sum(G.comm[g], s);
      PeerSum peer_sum(G.comm[g], s, peer ? &G.peer[g] : nullptr);
      NcclSum& ar = peer ? static_cast<NcclSum&>(peer_sum) : nccl_sum;
      ar.sum(rowsum.p, n);
      launch_row_shift(Z.p, n, nc, ld, rowsum.p, 1.0 / static_cast<double>(n), s);
      cudaEvent_t e0, e1;
      GBM_CUDA(cudaEventCreate(&e0));
      GBM_CUDA(cudaEventCreate(&e1));
      GBM_CUDA(cudaEventRecord(e0, s));
      double theta = 0.0;
      int it = 0;
      const bool okc = lanczos_top_singular_sharded(Z.p, n, nc, ld, &ar, 1e-13, 3000, x.p, &theta, &it, st.sm_count, s);
      GBM_CUDA(cudaEventRecord(e1, s));
      GBM_CUDA(cudaStreamSynchronize(s));
      float ms = 0.f;
      cudaEventElapsedTime(&ms, e0, e1);
      cudaEventDestroy(e0);
      cudaEventDestroy(e1);
      if (peer) {
        int perr = 0;
        GBM_CUDA(cudaMemcpy(&perr, G.peer[g].mb.error, sizeof(int), cudaMemcpyDeviceToHost));
        if (perr) GBM_THROW(GBM_ERR_RUNTIME, "gbm_sharded_kstd_pc1: a GPU of the group did not reach the peer-memory all-reduce in time");
      }
      eig[g] = ms;
      conv[g] = okc ? 1 : 0;
      iters[g] = it;
      if (launches) launches[g] += 8 + (peer ? 6 : 7) * it;
      if (okc && g == 0 && pc1_host) {
        GBM_CUDA(cudaMemcpyAsync(pc1_host, x.p, sizeof(double) * n, cudaMemcpyDeviceToHost, s));
        GBM_CUDA(cudaStreamSynchronize(s));
      }
    });
    // every rank sees the same bits from the all-reduces, so they all converge (or not) together
    if (conv[0]) {
      if (steps) *steps = iters[0];
      return *std::max_element(eig.begin(), eig.end());
    }
  }
  // one GPU, a small n, or no convergence: the single-GPU routine on every GPU (deterministic, no exchange)
  G.run([&](int g) {
    std::vector<double> tmp;
    double* out = pc1_host;
    if (g != 0 || !pc1_host) {
      tmp.resize(n);
      out = tmp.data();
    }
    double ms = 0.0;
    ok(gbm_kstd_pc1(m->dK[g], n, nullptr, out, &ms));
    eig[g] = ms;
    if (launches) launches[g] += state().launches;
  });
  if (steps) *steps = 0;
  return *std::max_element(eig.begin(), eig.end());
}

struct ScanOut {
  double *beta, *se, *stat, *nlp, *mean, *sd;
  uint8_t* keep;
};

// device results of one block, alive from the compute phase to the gather (released on the GPU's own thread)
struct BlockBufs {
  std::unique_ptr<Dev<double>> d[6];
  std::unique_ptr<Dev<uint8_t>> keep;
  std::unique_ptr<Dev<int64_t>> idx;
  void reset() {
    for (auto& x : d) x.reset();
    keep.reset();
    idx.reset();
  }
};
template <typename T>
T* ptr_of(const std::unique_ptr<Dev<T>>& b) {
  return b ? b->p : nullptr;
}

// marker loop on every block, results gathered into full-length host arrays.  Returns the slowest GPU's
// streaming-kernel time; *scan_ms / *gather_ms get the wall times of the two steps.
double sharded_scan(gbm_sharded* m, const double* Y, int64_t T, int64_t ldy, const double* C, int64_t k, int64_t ldc, int model,
                    int flags, const ScanOut& o, double* scan_ms, double* gather_ms, int64_t* launches) {
  gbm_group& G = *m->grp;
  const int64_t p = m->p;
  std::vector<double> kern(G.n_local, 0.0);
  std::vector<BlockBufs> buf(G.n_local);
  double* const want[6] = {o.beta, o.se, o.stat, o.nlp, o.mean, o.sd};
  const double t0 = now_ms();
  try {
    G.phase([&](int g) {
      const int64_t pc = m->ncols[G.rank_of(g)];
      BlockBufs& b = buf[g];
      for (int i = 0; i < 6; ++i)
        if (want[i]) b.d[i].reset(new Dev<double>(static_cast<size_t>(pc) * (i < 4 ? T : 1)));
      if (o.keep) b.keep.reset(new Dev<uint8_t>(pc));
      ok(gbm_scan(m->local[g], Y, T, ldy, C, k, ldc, model, flags, ptr_of(b.d[0]), ptr_of(b.d[1]), ptr_of(b.d[2]),
                  ptr_of(b.d[3]), ptr_of(b.d[4]), ptr_of(b.d[5]), ptr_of(b.keep)));
      kern[g] = state().main_ms;
      if (launches) launches[g] += state().launches;
    });
    const double t1 = now_ms();
    G.run([&](int g) {
      BlockBufs& b = buf[g];
      for (int i = 0; i < 6; ++i) gather_rows(G, g, ptr_of(b.d[i]), m->ncols, m->col0, p, i < 4 ? T : int64_t(1), want[i]);
      gather_rows(G, g, ptr_of(b.keep), m->ncols, m->col0, p, int64_t(1), o.keep);
      GBM_CUDA(cudaStreamSynchronize(state().stream));
      b.reset();
    });
    if (scan_ms) *scan_ms = t1 - t0;
    if (gather_ms) *gather_ms = now_ms() - t1;
  } catch (...) {
    try {
      G.run([&](int g) { buf[g].reset(); });
    } catch (...) {
    }
    throw;
  }
  return *std::max_element(kern.begin(), kern.end());
}

struct ColstatsOut {
  double *mean, *sd, *minnz;
  uint8_t* keep;
  int64_t* idx_cols;
};

// fixed-locus filter + ploidy probe on every block; returns (l, min over kept columns of the smallest nonzero value)
std::pair<int64_t, double> sharded_colstats(gbm_sharded* m, const ColstatsOut& o, int64_t* launches) {
  gbm_group& G = *m->grp;
  const int64_t p = m->p;
  std::vector<int64_t> kept(G.n_local, 0);
  std::vector<std::vector<double>> mink(G.n_local, std::vector<double>(1, 0.0));
  std::vector<BlockBufs> buf(G.n_local);
  double* const want[3] = {o.mean, o.sd, o.minnz};
  try {
    G.phase([&](int g) {
      const int64_t pc = m->ncols[G.rank_of(g)];
      BlockBufs& b = buf[g];
      for (int i = 0; i < 3; ++i)
        if (want[i]) b.d[i].reset(new Dev<double>(pc));
      if (o.keep) b.keep.reset(new Dev<uint8_t>(pc));
      b.idx.reset(new Dev<int64_t>(pc));
      double mk = 0.0;
      ok(gbm_colstats(m->local[g], ptr_of(b.d[0]), ptr_of(b.d[1]), ptr_of(b.d[2]), ptr_of(b.keep), b.idx->p, &kept[g], &mk));
      mink[g][0] = mk > 0.0 ? mk : 1e300;  // no kept column with a nonzero entry
      if (launches) launches[g] += state().launches;
    });
    // idx_cols = shard-order concatenation, every block's 1-based indices shifted by its first column
    const std::vector<int64_t> counts = G.all_counts(kept), offs = prefix(counts);
    const int64_t l = offs.back() + counts.back();
    G.reduce_host(mink, ncclMin);
    G.run([&](int g) {
      cudaStream_t s = state().stream;
      const int r = G.rank_of(g);
      BlockBufs& b = buf[g];
      for (int i = 0; i < 3; ++i) gather_rows(G, g, ptr_of(b.d[i]), m->ncols, m->col0, p, int64_t(1), want[i]);
      gather_rows(G, g, ptr_of(b.keep), m->ncols, m->col0, p, int64_t(1), o.keep);
      if (o.idx_cols) {
        if (counts[r] > 0)
          add_offset_kernel<<<static_cast<unsigned>((counts[r] + 255) / 256), 256, 0, s>>>(b.idx->p, counts[r], m->col0[r]);
        gather_rows(G, g, b.idx->p, counts, offs, l, int64_t(1), o.idx_cols);
      }
      GBM_CUDA(cudaStreamSynchronize(s));
      b.reset();
    });
    return {l, mink[0][0] >= 1e300 ? 0.0 : mink[0][0]};
  } catch (...) {
    try {
      G.run([&](int g) { buf[g].reset(); });
    } catch (...) {
    }
    throw;
  }
}

void check_lmm_covariates(int64_t n, const double* C, int64_t k, int64_t ldc, const char* who) {
  if (n < 4) GBM_THROW(GBM_ERR_ARGUMENT, std::string(who) + ": at least 4 entries are needed");
  if (n > 2147483647) GBM_THROW(GBM_ERR_ARGUMENT, "n too large for cuSOLVER");
  if (k < 0 || k > 2 || (k > 0 && (!C || ldc < n)))
    GBM_THROW(GBM_ERR_ARGUMENT, std::string(who) + ": 0..2 covariates besides the intercept are supported");
}

}  // namespace

struct gbm_sharded_lmm_plan {
  gbm_group* grp = nullptr;
  int64_t n = 0;
  std::vector<gbm_lmm_plan*> local;  // per local GPU; the same bits on every GPU of the group
  double eig_ms = 0.0;               // rank 0's syevd
};

namespace {

void free_lmm_plan(gbm_sharded_lmm_plan* P) {
  try {
    P->grp->run([&](int g) {
      if (!P->local[g]) return;
      cudaStreamSynchronize(state().stream);
      lmm_plan_destroy(P->local[g]);
      P->local[g] = nullptr;
    });
  } catch (...) {
  }
}

struct LmmFactorTimes {
  double kprep_ms = 0, eig_ms = 0, broadcast_ms = 0;
};

// The eigendecomposition, once per group.  Every GPU allocates its plan, and rank 0 puts K into its U buffer
// (load_k(plan, g), which may also transform it, *kprep_ms = its host time) and factors it, all in ONE G.phase: a
// failure there (an allocation, syevd info != 0) is agreed on by every rank before the first broadcast, so nobody
// waits in NCCL for a rank that has already returned.  Then U (ldu x n, padding included), S, U'y, U'[1, C] and the
// scalars travel from rank 0 to everybody.
gbm_sharded_lmm_plan* sharded_lmm_factor(gbm_group& G, int64_t n, const std::function<void(gbm_lmm_plan*, int)>& load_k,
                                         const double* y, const double* C, int64_t k, int64_t ldc, LmmFactorTimes* t,
                                         int64_t* launches) {
  std::unique_ptr<gbm_sharded_lmm_plan> P(new gbm_sharded_lmm_plan);
  P->grp = &G;
  P->n = n;
  P->local.assign(G.n_local, nullptr);
  std::vector<std::unique_ptr<Dev<double>>> scal(G.n_local);  // lam0, s_min, eig_ms, kprep_ms
  std::vector<std::array<double, 4>> h(G.n_local, std::array<double, 4>{0.0, 0.0, 0.0, 0.0});
  try {
    const double t0 = now_ms();
    G.phase([&](int g) {
      scal[g].reset(new Dev<double>(4));
      P->local[g] = lmm_plan_alloc(n, static_cast<int>(k) + 1);
      if (G.rank_of(g) != 0) return;
      gbm_lmm_plan* pl = P->local[g];
      const int64_t l0 = state().launches;
      const double tk = now_ms();
      load_k(pl, g);
      GBM_CUDA(cudaStreamSynchronize(state().stream));
      h[g][3] = now_ms() - tk;
      lmm_plan_factor(pl, y, C, k, ldc, &h[g][2]);
      h[g][0] = pl->lam0;
      h[g][1] = pl->s_min;
      if (launches) launches[g] += state().launches - l0;
    });
    const double t1 = now_ms();
    G.run([&](int g) {
      gbm_lmm_plan* pl = P->local[g];
      cudaStream_t s = state().stream;
      double* sc = scal[g]->p;
      if (G.rank_of(g) == 0) GBM_CUDA(cudaMemcpyAsync(sc, h[g].data(), sizeof(double) * 4, cudaMemcpyHostToDevice, s));
      if (G.world > 1) {
        GBM_NCCL(nccl().GroupStart());
        GBM_NCCL(nccl().Broadcast(pl->dU, pl->dU, static_cast<size_t>(pl->ldu) * n, ncclDouble, 0, G.comm[g], s));
        GBM_NCCL(nccl().Broadcast(pl->dS, pl->dS, static_cast<size_t>(n), ncclDouble, 0, G.comm[g], s));
        GBM_NCCL(nccl().Broadcast(pl->dYr, pl->dYr, static_cast<size_t>(n), ncclDouble, 0, G.comm[g], s));
        GBM_NCCL(nccl().Broadcast(pl->dCr, pl->dCr, static_cast<size_t>(n) * pl->Q0, ncclDouble, 0, G.comm[g], s));
        GBM_NCCL(nccl().Broadcast(sc, sc, 4, ncclDouble, 0, G.comm[g], s));
        GBM_NCCL(nccl().GroupEnd());
      }
      GBM_CUDA(cudaMemcpyAsync(h[g].data(), sc, sizeof(double) * 4, cudaMemcpyDeviceToHost, s));
      GBM_CUDA(cudaStreamSynchronize(s));
      pl->lam0 = h[g][0];
      pl->s_min = h[g][1];
      scal[g].reset();
    });
    if (t) {
      t->kprep_ms = h[0][3];
      t->eig_ms = (t1 - t0) - h[0][3];
      t->broadcast_ms = now_ms() - t1;
    }
  } catch (...) {
    try {
      G.run([&](int g) { scal[g].reset(); });
    } catch (...) {
    }
    free_lmm_plan(P.get());
    throw;
  }
  P->eig_ms = h[0][2];
  return P.release();
}

struct LmmOut {
  double *beta, *se, *stat, *nlp, *log_delta;
};

// the marker loop: every GPU runs gbm_lmm_plan_run on its own block (rotation in column blocks + delta search), then
// the five per-marker outputs are gathered in locus order.  Fills the marker fields of *t.
void sharded_lmm_run(gbm_sharded_lmm_plan* P, gbm_sharded* m, int flags, const LmmOut& o, gbm_reml_timing* t,
                     int64_t* launches) {
  gbm_group& G = *m->grp;
  const int64_t p = m->p;
  std::vector<std::vector<double>> dev_ms(G.n_local, std::vector<double>(2, 0.0));  // rotation, search
  std::vector<BlockBufs> buf(G.n_local);
  double* const want[5] = {o.beta, o.se, o.stat, o.nlp, o.log_delta};
  const double t0 = now_ms();
  try {
    G.phase([&](int g) {
      const int64_t pc = m->ncols[G.rank_of(g)];
      BlockBufs& b = buf[g];
      for (int i = 0; i < 5; ++i)
        if (want[i]) b.d[i].reset(new Dev<double>(pc));
      double tflops = 0.0, search_ms = 0.0;
      ok(gbm_lmm_plan_run(P->local[g], m->local[g], flags, ptr_of(b.d[0]), ptr_of(b.d[1]), ptr_of(b.d[2]), ptr_of(b.d[3]),
                          ptr_of(b.d[4]), &tflops, &search_ms));
      dev_ms[g][0] = state().main_ms;  // the rotation GEMMs' events
      dev_ms[g][1] = search_ms;
      if (launches) launches[g] += state().launches;
    });
    const double t1 = now_ms();
    G.run([&](int g) {
      BlockBufs& b = buf[g];
      for (int i = 0; i < 5; ++i) gather_rows(G, g, ptr_of(b.d[i]), m->ncols, m->col0, p, int64_t(1), want[i]);
      GBM_CUDA(cudaStreamSynchronize(state().stream));
      b.reset();
    });
    t->scan_ms = t1 - t0;
    t->gather_ms = now_ms() - t1;
  } catch (...) {
    try {
      G.run([&](int g) { buf[g].reset(); });
    } catch (...) {
    }
    throw;
  }
  G.reduce_host(dev_ms, ncclMax);  // the slowest GPU
  t->rotation_ms = dev_ms[0][0];
  t->search_ms = dev_ms[0][1];
  t->rotation_tflops = 2.0 * static_cast<double>(m->n) * static_cast<double>(m->n) * static_cast<double>(p) /
                       (t->rotation_ms * 1e-3) / 1e12;
  t->n_gpus = G.world;
}

void check_lmm_plan(const gbm_sharded_lmm_plan* P, const gbm_sharded* m) {
  if (!P) GBM_THROW(GBM_ERR_ARGUMENT, "gbm_sharded_lmm_plan_run: null plan");
  if (P->grp != m->grp) GBM_THROW(GBM_ERR_ARGUMENT, "gbm_sharded_lmm_plan_run: the plan belongs to another group");
  if (P->n != m->n)
    GBM_THROW(GBM_ERR_ARGUMENT, "gbm_sharded_lmm_plan_run: the matrix and the GRM have different numbers of entries");
}

}  // namespace

#define GBM_GROUP_BEGIN try {
#define GBM_GROUP_END                                  \
  }                                                    \
  catch (const gbm::Error& e) {                        \
    set_error(e.msg);                                  \
    return e.code;                                     \
  }                                                    \
  catch (const std::exception& e) {                    \
    set_error(std::string("internal: ") + e.what());   \
    return GBM_ERR_RUNTIME;                            \
  }                                                    \
  return GBM_OK;

extern "C" {

int gbm_group_create_local(int n_gpus, const int* devices, gbm_group** out) {
  GBM_GROUP_BEGIN
  if (!out) GBM_THROW(GBM_ERR_ARGUMENT, "gbm_group_create_local: null output");
  int count = 0;
  if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0)
    GBM_THROW(GBM_ERR_CUDA, "no CUDA device: libgbm_b200 has no CPU fallback");
  if (n_gpus < 1 || n_gpus > count)
    GBM_THROW(GBM_ERR_ARGUMENT, "gbm_group_create_local: " + std::to_string(n_gpus) + " GPUs requested, " + std::to_string(count) + " visible");
  std::vector<int> dev(n_gpus);
  for (int g = 0; g < n_gpus; ++g) {
    dev[g] = devices ? devices[g] : g;
    if (dev[g] < 0 || dev[g] >= count) GBM_THROW(GBM_ERR_ARGUMENT, "gbm_group_create_local: device index out of range");
    for (int h = 0; h < g; ++h)
      if (dev[h] == dev[g]) GBM_THROW(GBM_ERR_ARGUMENT, "gbm_group_create_local: a device is listed twice");
  }
  std::unique_ptr<gbm_group> G(new gbm_group);
  G->world = G->n_local = n_gpus;
  G->first_rank = 0;
  G->threaded = true;
  for (int g = 0; g < n_gpus; ++g) {
    G->owned.emplace_back(new State);
    G->ctx.push_back(G->owned.back().get());
    G->workers.emplace_back(new Worker);
    G->workers.back()->start(G->ctx.back());
  }
  try {
    G->run([&](int g) { init_state(state(), dev[g]); });
    int cur = 0;
    cudaGetDevice(&cur);
    G->comm.assign(n_gpus, nullptr);
    GBM_NCCL(nccl().CommInitAll(G->comm.data(), n_gpus, dev.data()));
    cudaSetDevice(cur);
  } catch (...) {
    for (auto& w : G->workers) w->stop();
    throw;
  }
  *out = G.release();
  GBM_GROUP_END
}

int gbm_group_unique_id(void* id) {
  GBM_GROUP_BEGIN
  if (!id) GBM_THROW(GBM_ERR_ARGUMENT, "gbm_group_unique_id: null output");
  static_assert(sizeof(ncclUniqueId) == GBM_GROUP_ID_BYTES, "ncclUniqueId is 128 bytes");
  ncclUniqueId u;
  GBM_NCCL(nccl().GetUniqueId(&u));
  memcpy(id, &u, sizeof(u));
  GBM_GROUP_END
}

int gbm_group_create_rank(const void* id, int world, int rank, gbm_group** out) {
  GBM_GROUP_BEGIN
  if (!id || !out) GBM_THROW(GBM_ERR_ARGUMENT, "gbm_group_create_rank: null pointer");
  if (world < 1 || rank < 0 || rank >= world) GBM_THROW(GBM_ERR_ARGUMENT, "gbm_group_create_rank: rank out of range");
  require_ready();  // the GPU is the one gbm_init selected on this process
  std::unique_ptr<gbm_group> G(new gbm_group);
  G->world = world;
  G->n_local = 1;
  G->first_rank = rank;
  G->threaded = false;
  G->ctx.push_back(&state());
  ncclUniqueId u;
  memcpy(&u, id, sizeof(u));
  G->comm.assign(1, nullptr);
  GBM_NCCL(nccl().CommInitRank(&G->comm[0], world, u, rank));
  *out = G.release();
  GBM_GROUP_END
}

int gbm_group_info(const gbm_group* g, int* world, int* n_local, int* first_rank) {
  GBM_GROUP_BEGIN
  check_group(g);
  if (world) *world = g->world;
  if (n_local) *n_local = g->n_local;
  if (first_rank) *first_rank = g->first_rank;
  GBM_GROUP_END
}

int gbm_group_free(gbm_group* g) {
  GBM_GROUP_BEGIN
  if (!g) return GBM_OK;
  {
    std::lock_guard<std::mutex> lk(g->mutex);
    free_peer(*g);
    for (ncclComm_t c : g->comm)
      if (c) nccl().CommDestroy(c);
    if (g->threaded) {
      try {
        g->run([&](int) { shutdown_state(state()); });
      } catch (...) {
      }
      for (auto& w : g->workers) w->stop();
    }
  }
  delete g;
  GBM_GROUP_END
}

static gbm_sharded* new_sharded(gbm_group* g, int64_t n) {
  gbm_sharded* m = new gbm_sharded;
  m->grp = g;
  m->n = n;
  m->local.assign(g->n_local, nullptr);
  m->dK.assign(g->n_local, nullptr);
  return m;
}

int gbm_sharded_upload(gbm_group* g, const double* A, int64_t n, int64_t p, int64_t lda, int compact, gbm_sharded** out,
                       int* packed) {
  GBM_GROUP_BEGIN
  check_group(g);
  if (!A || !out) GBM_THROW(GBM_ERR_ARGUMENT, "gbm_sharded_upload: null pointer");
  if (n < 2 || lda < n) GBM_THROW(GBM_ERR_ARGUMENT, "gbm_sharded_upload: bad matrix shape");
  if (p < g->world) GBM_THROW(GBM_ERR_ARGUMENT, "gbm_sharded_upload: fewer markers than GPUs");
  std::lock_guard<std::mutex> lk(g->mutex);
  std::unique_ptr<gbm_sharded> m(new_sharded(g, n));
  gbm_group& G = *g;
  std::vector<std::vector<double>> pk(G.n_local, std::vector<double>(1, 0.0));
  auto bounds = [&](int r, int64_t* j0, int64_t* pc) {
    *j0 = p * r / G.world;
    *pc = p * (r + 1) / G.world - *j0;
  };
  try {
    G.phase([&](int gi) {
      int64_t j0, pc;
      bounds(G.rank_of(gi), &j0, &pc);
      int is_packed = 0;
      if (compact)
        ok(gbm_matrix_upload_compact(A + j0 * lda, n, pc, lda, &m->local[gi], &is_packed));
      else
        ok(gbm_matrix_upload(A + j0 * lda, n, pc, lda, &m->local[gi]));
      pk[gi][0] = is_packed;
    });
    std::vector<std::vector<double>> all = pk;
    G.reduce_host(all, ncclMin);
    m->packed = all[0][0] > 0.5 ? 1 : 0;
    if (compact && !m->packed)  // some block is not dosage data: Float64 slabs everywhere
      G.phase([&](int gi) {
        if (pk[gi][0] < 0.5) return;
        int64_t j0, pc;
        bounds(G.rank_of(gi), &j0, &pc);
        gbm_matrix_free(m->local[gi]);
        m->local[gi] = nullptr;
        ok(gbm_matrix_upload(A + j0 * lda, n, pc, lda, &m->local[gi]));
      });
    finish_layout(m.get());
  } catch (...) {
    try {
      free_blocks(m.get());
    } catch (...) {
    }
    throw;
  }
  if (packed) *packed = m->packed;
  *out = m.release();
  GBM_GROUP_END
}

int gbm_sharded_generate(gbm_group* g, uint64_t seed, int64_t n, int64_t p, int kind, int pack, gbm_sharded** out,
                         int* packed) {
  GBM_GROUP_BEGIN
  check_group(g);
  if (!out) GBM_THROW(GBM_ERR_ARGUMENT, "gbm_sharded_generate: null pointer");
  if (p < g->world) GBM_THROW(GBM_ERR_ARGUMENT, "gbm_sharded_generate: fewer markers than GPUs");
  std::lock_guard<std::mutex> lk(g->mutex);
  std::unique_ptr<gbm_sharded> m(new_sharded(g, n));
  gbm_group& G = *g;
  std::vector<gbm_matrix*> codes(G.n_local, nullptr);
  std::vector<std::vector<double>> pk(G.n_local, std::vector<double>(1, 0.0));
  try {
    G.phase([&](int gi) {
      const int r = G.rank_of(gi);
      const int64_t j0 = p * r / G.world, pc = p * (r + 1) / G.world - j0;
      ok(gbm_matrix_generate(seed, n, pc, j0, kind, &m->local[gi]));
      if (pack) {
        int64_t bad = 0;
        ok(gbm_matrix_pack(m->local[gi], &codes[gi], &bad));
        pk[gi][0] = codes[gi] ? 1.0 : 0.0;
      }
    });
    if (pack) {
      std::vector<std::vector<double>> all = pk;
      G.reduce_host(all, ncclMin);
      m->packed = all[0][0] > 0.5 ? 1 : 0;
      G.run([&](int gi) {
        if (m->packed) {
          gbm_matrix_free(m->local[gi]);
          m->local[gi] = codes[gi];
        } else if (codes[gi]) {
          gbm_matrix_free(codes[gi]);
        }
        codes[gi] = nullptr;
      });
    }
    finish_layout(m.get());
  } catch (...) {
    try {
      G.run([&](int gi) {
        if (codes[gi]) gbm_matrix_free(codes[gi]);
      });
      free_blocks(m.get());
    } catch (...) {
    }
    throw;
  }
  if (packed) *packed = m->packed;
  *out = m.release();
  GBM_GROUP_END
}

int gbm_sharded_adopt(gbm_group* g, gbm_matrix* const* local, gbm_sharded** out) {
  GBM_GROUP_BEGIN
  check_group(g);
  if (!local || !out) GBM_THROW(GBM_ERR_ARGUMENT, "gbm_sharded_adopt: null pointer");
  std::lock_guard<std::mutex> lk(g->mutex);
  int64_t n = 0;
  for (int i = 0; i < g->n_local; ++i) {
    if (!local[i]) GBM_THROW(GBM_ERR_ARGUMENT, "gbm_sharded_adopt: null block handle");
    int64_t ni = 0;
    ok(gbm_matrix_info(local[i], &ni, nullptr, nullptr, nullptr));
    if (i && ni != n) GBM_THROW(GBM_ERR_ARGUMENT, "gbm_sharded_adopt: blocks with different numbers of entries");
    n = ni;
  }
  std::unique_ptr<gbm_sharded> m(new_sharded(g, n));
  m->owned = false;
  for (int i = 0; i < g->n_local; ++i) m->local[i] = local[i];
  finish_layout(m.get());
  *out = m.release();
  GBM_GROUP_END
}

int gbm_sharded_info(const gbm_sharded* m, int64_t* n, int64_t* p, int64_t* first_col, int64_t* ncols, int* packed) {
  GBM_GROUP_BEGIN
  check_sharded(m);
  if (n) *n = m->n;
  if (p) *p = m->p;
  for (int g = 0; g < m->grp->n_local; ++g) {
    if (first_col) first_col[g] = m->col0[m->grp->rank_of(g)];
    if (ncols) ncols[g] = m->ncols[m->grp->rank_of(g)];
  }
  if (packed) *packed = m->packed;
  GBM_GROUP_END
}

int gbm_sharded_free(gbm_sharded* m) {
  GBM_GROUP_BEGIN
  if (!m) return GBM_OK;
  if (m->grp) {
    std::lock_guard<std::mutex> lk(m->grp->mutex);
    free_blocks(m);
  }
  delete m;
  GBM_GROUP_END
}

int gbm_sharded_colstats(gbm_sharded* m, double* mean, double* sd, double* min_nonzero, uint8_t* keep, int64_t* idx_cols,
                         int64_t* n_keep, double* min_nonzero_kept) {
  GBM_GROUP_BEGIN
  check_sharded(m);
  std::lock_guard<std::mutex> lk(m->grp->mutex);
  const auto r = sharded_colstats(m, ColstatsOut{mean, sd, min_nonzero, keep, idx_cols}, nullptr);
  if (n_keep) *n_keep = r.first;
  if (min_nonzero_kept) *min_nonzero_kept = r.second;
  GBM_GROUP_END
}

int gbm_sharded_grm(gbm_sharded* m, int grm_type, int ploidy, int flags, double* K, double* tflops) {
  GBM_GROUP_BEGIN
  check_sharded(m);
  std::lock_guard<std::mutex> lk(m->grp->mutex);
  const GrmTimes t = sharded_grm(m, grm_type, ploidy, flags, nullptr);
  if (tflops)
    *tflops = static_cast<double>(m->n) * static_cast<double>(m->n + 1) * static_cast<double>(m->p) /
              ((t.grm_ms + t.allreduce_ms) * 1e-3) / 1e12;
  if (K)
    m->grp->run([&](int g) {
      if (g != 0) return;
      GBM_CUDA(cudaMemcpyAsync(K, m->dK[0], sizeof(double) * m->n * m->n, cudaMemcpyDeviceToHost, state().stream));
      GBM_CUDA(cudaStreamSynchronize(state().stream));
    });
  GBM_GROUP_END
}

int gbm_sharded_kstd_pc1(gbm_sharded* m, const double* K, double* pc1, double* eig_ms) {
  GBM_GROUP_BEGIN
  check_sharded(m);
  if (!pc1) GBM_THROW(GBM_ERR_ARGUMENT, "gbm_sharded_kstd_pc1: null output");
  std::lock_guard<std::mutex> lk(m->grp->mutex);
  if (K) {
    m->grp->run([&](int g) {
      ensure_dK(m, g);
      GBM_CUDA(cudaMemcpyAsync(m->dK[g], K, sizeof(double) * m->n * m->n, cudaMemcpyDefault, state().stream));
      GBM_CUDA(cudaStreamSynchronize(state().stream));
    });
    m->have_K = true;
  }
  const double ms = sharded_kstd_pc1(m, pc1, nullptr, nullptr);
  if (eig_ms) *eig_ms = ms;
  GBM_GROUP_END
}

int gbm_sharded_scan(gbm_sharded* m, const double* Y, int64_t T, int64_t ldy, const double* C, int64_t k, int64_t ldc,
                     int model, int flags, double* beta, double* se, double* stat, double* neglog10p, double* mean,
                     double* sd, uint8_t* keep) {
  GBM_GROUP_BEGIN
  check_sharded(m);
  std::lock_guard<std::mutex> lk(m->grp->mutex);
  sharded_scan(m, Y, T, ldy, C, k, ldc, model, flags, ScanOut{beta, se, stat, neglog10p, mean, sd, keep}, nullptr, nullptr,
               nullptr);
  GBM_GROUP_END
}

int gbm_sharded_gwas(gbm_sharded* m, const double* y, int model, int grm_type, int flags, double* stat, double* beta,
                     double* se, double* neglog10p, double* mean, double* sd, uint8_t* keep, int64_t* idx_cols,
                     int64_t* n_keep, double* pc1, gbm_gwas_timing* timing) {
  GBM_GROUP_BEGIN
  check_sharded(m);
  if (!y) GBM_THROW(GBM_ERR_ARGUMENT, "gbm_sharded_gwas: null trait vector");
  if (grm_type != GBM_GRM_SIMPLE && grm_type != GBM_GRM_PLOIDY_AWARE)
    GBM_THROW(GBM_ERR_ARGUMENT, "Unrecognised `GRM_type`. Please select from:\n\t‣ simple\n\t‣ ploidy-aware");
  gbm_group& G = *m->grp;
  std::lock_guard<std::mutex> lk(G.mutex);
  std::vector<int64_t> launches(G.n_local, 0);
  gbm_gwas_timing t;
  memset(&t, 0, sizeof(t));
  const double t0 = now_ms();
  // v = std(G, dims=1); idx_cols; minimum(G[G .!= 0])   (gwas.jl:112-113, :119)
  const auto cs = sharded_colstats(m, ColstatsOut{nullptr, nullptr, nullptr, nullptr, idx_cols}, launches.data());
  if (n_keep) *n_keep = cs.first;
  int ploidy = 2;
  if (grm_type == GBM_GRM_PLOIDY_AWARE) {
    if (!(cs.second > 0.0)) GBM_THROW(GBM_ERR_RUNTIME, "cannot infer the ploidy: no non-zero allele frequency among the kept loci");
    ploidy = static_cast<int>(nearbyint(1.0 / cs.second));  // Int(round(1 / minimum(G[G .!= 0.0])))
  }
  t.ploidy = ploidy;
  const double t1 = now_ms();
  t.colstats_ms = t1 - t0;
  // GRM on all entries and loci (gwas.jl:117-126)
  const GrmTimes gt = sharded_grm(m, grm_type, ploidy, flags & GBM_GRM_NO_CENTRE, launches.data());
  t.grm_ms = gt.grm_ms;
  t.allreduce_ms = gt.allreduce_ms;
  t.grm_tflops = static_cast<double>(m->n) * static_cast<double>(m->n + 1) * static_cast<double>(m->p) /
                 ((gt.grm_ms + gt.allreduce_ms) * 1e-3) / 1e12;
  const double t2 = now_ms();
  // K standardisation (gwas.jl:130) and PC1 (:234, :357)
  std::vector<double> pc(static_cast<size_t>(m->n));
  int steps = 0;
  t.eig_ms = sharded_kstd_pc1(m, pc.data(), &steps, launches.data());
  t.lanczos_steps = steps;
  if (pc1) memcpy(pc1, pc.data(), sizeof(double) * m->n);
  const double t3 = now_ms();
  t.kstd_pc1_ms = t3 - t2;
  // marker loop with X = [1, PC1, g_j]  (gwas.jl:239-249 / :363-389)
  t.scan_kernel_ms = sharded_scan(m, y, 1, m->n, pc.data(), 1, m->n, model, flags & GBM_PVALUE_TWO_SIDED,
                                  ScanOut{beta, se, stat, neglog10p, mean, sd, keep}, &t.scan_ms, &t.gather_ms, launches.data());
  t.total_ms = now_ms() - t0;
  for (int64_t l : launches) t.launches += l;
  if (timing) *timing = t;
  GBM_GROUP_END
}


int gbm_sharded_lmm_plan_create(gbm_sharded* m, const double* K, const double* y, const double* C, int64_t k,
                                int64_t ldc, gbm_sharded_lmm_plan** plan, double* eig_ms, double* null_log_delta) {
  GBM_GROUP_BEGIN
  check_sharded(m);
  if (!K || !y || !plan) GBM_THROW(GBM_ERR_ARGUMENT, "gbm_sharded_lmm_plan_create: null pointer");
  check_lmm_covariates(m->n, C, k, ldc, "gbm_sharded_lmm_plan_create");
  std::lock_guard<std::mutex> lk(m->grp->mutex);
  const int64_t n = m->n;
  gbm_sharded_lmm_plan* P = sharded_lmm_factor(
      *m->grp, n, [&](gbm_lmm_plan* pl, int) { lmm_plan_load_k(pl, K, n); }, y, C, k, ldc, nullptr, nullptr);
  if (eig_ms) *eig_ms = P->eig_ms;
  if (null_log_delta) *null_log_delta = P->local[0]->lam0;
  *plan = P;
  GBM_GROUP_END
}

int gbm_sharded_lmm_plan_run(gbm_sharded_lmm_plan* plan, gbm_sharded* m, int flags, double* beta, double* se,
                             double* stat, double* neglog10p, double* log_delta, gbm_reml_timing* timing) {
  GBM_GROUP_BEGIN
  check_sharded(m);
  check_lmm_plan(plan, m);
  std::lock_guard<std::mutex> lk(m->grp->mutex);
  std::vector<int64_t> launches(m->grp->n_local, 0);
  gbm_reml_timing t;
  memset(&t, 0, sizeof(t));
  const double t0 = now_ms();
  sharded_lmm_run(plan, m, flags, LmmOut{beta, se, stat, neglog10p, log_delta}, &t, launches.data());
  t.total_ms = now_ms() - t0;
  for (int64_t l : launches) t.launches += l;
  if (timing) *timing = t;
  GBM_GROUP_END
}

int gbm_sharded_lmm_plan_free(gbm_sharded_lmm_plan* plan) {
  GBM_GROUP_BEGIN
  if (!plan) return GBM_OK;
  {
    std::lock_guard<std::mutex> lk(plan->grp->mutex);
    free_lmm_plan(plan);
  }
  delete plan;
  GBM_GROUP_END
}

int gbm_sharded_gwasreml(gbm_sharded* m, const double* y, int grm_type, int flags, double* stat, double* beta,
                         double* se, double* neglog10p, double* log_delta, int64_t* idx_cols, int64_t* n_keep,
                         double* null_log_delta, gbm_reml_timing* timing) {
  GBM_GROUP_BEGIN
  check_sharded(m);
  if (!y) GBM_THROW(GBM_ERR_ARGUMENT, "gbm_sharded_gwasreml: null trait vector");
  if (grm_type != GBM_GRM_SIMPLE && grm_type != GBM_GRM_PLOIDY_AWARE)
    GBM_THROW(GBM_ERR_ARGUMENT, "Unrecognised `GRM_type`. Please select from:\n\t‣ simple\n\t‣ ploidy-aware");
  // one flags word for the scan only: the GRM is always centred (GBM_GRM_NO_CENTRE has the value of
  // GBM_PVALUE_TWO_SIDED, so it cannot be passed here)
  if (flags & ~(GBM_PVALUE_TWO_SIDED | GBM_LMM_REFERENCE_OBJECTIVE))
    GBM_THROW(GBM_ERR_ARGUMENT, "gbm_sharded_gwasreml: flags may only hold GBM_PVALUE_TWO_SIDED and GBM_LMM_REFERENCE_OBJECTIVE");
  check_lmm_covariates(m->n, nullptr, 0, m->n, "gbm_sharded_gwasreml");
  gbm_group& G = *m->grp;
  std::lock_guard<std::mutex> lk(G.mutex);
  const int64_t n = m->n;
  const bool ref = (flags & GBM_LMM_REFERENCE_OBJECTIVE) != 0;
  std::vector<int64_t> launches(G.n_local, 0);
  gbm_reml_timing t;
  memset(&t, 0, sizeof(t));
  const double t0 = now_ms();
  // v = std(G, dims=1); idx_cols; minimum(G[G .!= 0])   (gwas.jl:112-113, :119)
  const auto cs = sharded_colstats(m, ColstatsOut{nullptr, nullptr, nullptr, nullptr, idx_cols}, launches.data());
  if (n_keep) *n_keep = cs.first;
  int ploidy = 2;
  if (grm_type == GBM_GRM_PLOIDY_AWARE) {
    if (!(cs.second > 0.0)) GBM_THROW(GBM_ERR_RUNTIME, "cannot infer the ploidy: no non-zero allele frequency among the kept loci");
    ploidy = static_cast<int>(nearbyint(1.0 / cs.second));  // Int(round(1 / minimum(G[G .!= 0.0])))
  }
  t.ploidy = ploidy;
  t.colstats_ms = now_ms() - t0;
  // GRM on all entries and loci (gwas.jl:117-126), resident on every GPU
  const GrmTimes gt = sharded_grm(m, grm_type, ploidy, 0, launches.data());
  t.grm_ms = gt.grm_ms;
  t.allreduce_ms = gt.allreduce_ms;
  t.grm_tflops = static_cast<double>(n) * static_cast<double>(n + 1) * static_cast<double>(m->p) /
                 ((gt.grm_ms + gt.allreduce_ms) * 1e-3) / 1e12;
  // rank 0: K into the plan's U buffer; for the reference objective K = (K .- mean(K, dims=1)) ./ std(K, dims=1)
  // (gwas.jl:130, the kernels of gbm_kstd_pc1) and its symmetric part, the matrix a rotation can factor
  auto load_k = [&](gbm_lmm_plan* pl, int g) {
    lmm_plan_load_k(pl, m->dK[g], n);
    if (!ref) return;
    State& st = state();
    const int stride = scan_record_stride(0, true);
    Dev<double> rec(static_cast<size_t>(n) * stride), mean(n), sd(n);
    launch_scan_sums(pl->dU, n, n, pl->ldu, nullptr, 0, 0, true, rec.p, st.sm_count, st.stream);
    launch_colstats_finalize(rec.p, stride, n, n, mean.p, sd.p, nullptr, nullptr, st.stream);
    launch_k_standardise(pl->dU, n, n, pl->ldu, mean.p, sd.p, st.stream);
    launch_symmetrise(pl->dU, n, pl->ldu, st.stream);
    st.launches += 4;
  };
  LmmFactorTimes ft;
  std::unique_ptr<gbm_sharded_lmm_plan, int (*)(gbm_sharded_lmm_plan*)> P(
      sharded_lmm_factor(G, n, load_k, y, nullptr, 0, n, &ft, launches.data()), [](gbm_sharded_lmm_plan* q) {
        free_lmm_plan(q);
        delete q;
        return GBM_OK;
      });
  t.kprep_ms = ft.kprep_ms;
  t.eig_ms = ft.eig_ms;
  t.broadcast_ms = ft.broadcast_ms;
  if (null_log_delta) *null_log_delta = P->local[0]->lam0;
  // marker loop: rotation + delta search per GPU, gather in locus order (gwas.jl:586-607)
  sharded_lmm_run(P.get(), m, flags, LmmOut{beta, se, stat, neglog10p, log_delta}, &t, launches.data());
  t.total_ms = now_ms() - t0;
  for (int64_t l : launches) t.launches += l;
  if (timing) *timing = t;
  GBM_GROUP_END
}

}  // extern "C"
