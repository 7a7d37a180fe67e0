// bkid_dist.cuh -- the hot path over several GPUs, inside the library (SURVEY.md 8e).  Included by bkid_core.cu.
//
// One rank per GPU; every rank holds a contiguous slice of the coordinate-sorted record stream (genomic bins, in rank
// order) and calls bkid_dist_run collectively.  The exchanges are done HERE, through a small communicator interface:
//
//   NcclComm    NCCL (dlopen'ed libnccl.so.2): ncclAllReduce for the sums, grouped ncclSend / ncclRecv for the
//               all-to-all of candidate records / pairs and the all-gathers of clusters / evidence rows.  One rank per
//               process (bench.py under torchrun: the unique id travels through torch.distributed once) or one rank per
//               host thread of a single process (the BreakID driver with -gpu 0,1,...: ncclCommInitAll).
//   LocalComm   ranks = host threads of ONE process whose contexts may share a device: the exchanges are device copies
//               between the contexts behind a barrier.  This is how the sharded path is tested on a one-GPU box
//               (tests/test_gpu_parity.py: world sizes 2..5 against the oracle) -- no kernel ever waits on another rank.
//
//   stage                          exchange
//   -----------------------------  --------------------------------------------------------------------------------
//   classify + insert statistics   all-reduce (sum |isize|, count, sum isize^2; max |isize|)
//   truncating sd accumulator      one pass on all ranks at once + all-reduce (sum floor, #correctable); only if a record can
//                                  need a rounding correction: the exact replay chained rank to rank (point to point)
//   candidate records (48 B)       fused owner + stable partition kernel, counts exchange, all-to-all by name-hash owner
//   discordant pairs (64 B)        global bucket histogram all-reduce -> LPT bucket->rank table, partition, all-to-all
//   mask + clustering + summary    none (buckets are independent, src/BreakID.cc:119-167)
//   cluster summaries (192 B)      all-gather, ordered by (bucket name rank, cluster id)
//   split-read evidence rows       all-gather (coordinate order = rank order)
//   region coverage / bp depth     partial counts per shard, all-reduce (sum)
//   vote / AF / 41-mers            replicated (tiny)
#pragma once
#include <condition_variable>
#include <dlfcn.h>
#include <mutex>
#include <thread>

// ---------------------------------------------------------------------------------------------------------------
// communicators
// ---------------------------------------------------------------------------------------------------------------
enum BkOp { BK_SUM = 0, BK_MAX = 1 };
enum BkType { BK_U32 = 0, BK_U64 = 1 };

struct bkid_comm {
  int rank = 0, world = 1;
  std::string err;
  virtual ~bkid_comm() {}
  // in-place all-reduce of n elements on the device, ordered on stream st; complete (host-synchronised) on return
  virtual int allreduce(void *dev, int n, BkType ty, BkOp op, cudaStream_t st) = 0;
  // small host metadata: every rank contributes n values
  virtual int allgather_host(const uint64_t *mine, int n, uint64_t *all) = 0;
  // rows [send_off[r], send_off[r+1]) of `send` go to rank r; rows from rank s land at recv_off[s] (offsets in rows, [world+1])
  virtual int alltoallv(const void *send, const uint64_t *send_off, void *recv, const uint64_t *recv_off, int row_bytes, cudaStream_t st) = 0;
  // every rank's block of rows, in rank order, on every rank
  virtual int allgatherv(const void *send, uint64_t nrows, void *recv, const uint64_t *recv_off, int row_bytes, cudaStream_t st) = 0;
  // one int64 handed from rank `from` to rank `to` (the sd replay chain); other ranks return immediately
  virtual int relay_i64(long long *v, int from, int to) = 0;
  // this rank failed: release the ranks that wait for it (communicators that cannot do so leave it to the caller's timeout)
  virtual void abort() {}
};

// ---- ranks as threads of one process ----------------------------------------------------------------------------
struct LocalGroup {
  int world;
  std::mutex mu; std::condition_variable cv; int arrived = 0; unsigned long long gen = 0;
  bool aborted = false;                     // a rank failed: every barrier returns at once, every collective reports an error
  std::vector<const void *> ptr; std::vector<std::vector<uint64_t>> meta; std::vector<std::vector<unsigned long long>> host;
  long long relay = 0;
  explicit LocalGroup(int w) : world(w), ptr(w), meta(w), host(w) {}
  bool barrier()                            // false: the group was aborted
  {
    std::unique_lock<std::mutex> lk(mu);
    if (aborted) return false;
    unsigned long long g0 = gen;
    if (++arrived == world) { arrived = 0; ++gen; cv.notify_all(); }
    else cv.wait(lk, [&] { return gen != g0 || aborted; });
    return !aborted;
  }
  void abort()
  {
    std::lock_guard<std::mutex> lk(mu);
    aborted = true;
    cv.notify_all();
  }
};
struct LocalComm : bkid_comm {
  std::shared_ptr<LocalGroup> g;
  LocalComm(std::shared_ptr<LocalGroup> grp, int r) : g(std::move(grp)) { rank = r; world = g->world; }
  void abort() override { g->abort(); }
  int allreduce(void *dev, int n, BkType ty, BkOp op, cudaStream_t st) override
  {
    size_t es = ty == BK_U64 ? 8 : 4;
    std::vector<unsigned long long> &mine = g->host[rank];
    mine.assign((size_t)n, 0ull);
    std::vector<unsigned char> tmp((size_t)n * es);
    if (n) { if (cudaMemcpyAsync(tmp.data(), dev, (size_t)n * es, cudaMemcpyDeviceToHost, st) != cudaSuccess) return BKID_ERR_CUDA; cudaStreamSynchronize(st); }
    for (int i = 0; i < n; ++i) mine[i] = ty == BK_U64 ? ((unsigned long long *)tmp.data())[i] : ((unsigned *)tmp.data())[i];
    if (!g->barrier()) { err = "another rank failed"; return BKID_ERR_ARG; }
    std::vector<unsigned long long> acc((size_t)n, 0ull);
    for (int r = 0; r < world; ++r)
      for (int i = 0; i < n; ++i) acc[i] = op == BK_SUM ? acc[i] + g->host[r][i] : std::max(acc[i], g->host[r][i]);
    for (int i = 0; i < n; ++i) { if (ty == BK_U64) ((unsigned long long *)tmp.data())[i] = acc[i]; else ((unsigned *)tmp.data())[i] = (unsigned)acc[i]; }
    if (n) { if (cudaMemcpyAsync(dev, tmp.data(), (size_t)n * es, cudaMemcpyHostToDevice, st) != cudaSuccess) return BKID_ERR_CUDA; cudaStreamSynchronize(st); }
    if (!g->barrier()) { err = "another rank failed"; return BKID_ERR_ARG; }
    return 0;
  }
  int allgather_host(const uint64_t *mine, int n, uint64_t *all) override
  {
    g->meta[rank].assign(mine, mine + n);
    if (!g->barrier()) { err = "another rank failed"; return BKID_ERR_ARG; }
    for (int r = 0; r < world; ++r) for (int i = 0; i < n; ++i) all[(size_t)r * n + i] = g->meta[r][i];
    if (!g->barrier()) { err = "another rank failed"; return BKID_ERR_ARG; }
    return 0;
  }
  int alltoallv(const void *send, const uint64_t *send_off, void *recv, const uint64_t *recv_off, int row_bytes, cudaStream_t st) override
  {
    cudaStreamSynchronize(st);                               // my send buffer is complete before anybody reads it
    g->ptr[rank] = send;
    g->meta[rank].assign(send_off, send_off + world + 1);
    if (!g->barrier()) { err = "another rank failed"; return BKID_ERR_ARG; }
    for (int s = 0; s < world; ++s) {
      uint64_t a = g->meta[s][rank], b = g->meta[s][rank + 1];
      if (b > a && cudaMemcpyAsync((char *)recv + recv_off[s] * (size_t)row_bytes, (const char *)g->ptr[s] + a * (size_t)row_bytes, (b - a) * (size_t)row_bytes, cudaMemcpyDefault, st) != cudaSuccess)
        return BKID_ERR_CUDA;
    }
    cudaStreamSynchronize(st);
    g->barrier();                                            // every reader is done: send buffers may be reused
    return 0;
  }
  int allgatherv(const void *send, uint64_t nrows, void *recv, const uint64_t *recv_off, int row_bytes, cudaStream_t st) override
  {
    cudaStreamSynchronize(st);
    g->ptr[rank] = send;
    g->meta[rank].assign(1, nrows);
    if (!g->barrier()) { err = "another rank failed"; return BKID_ERR_ARG; }
    for (int s = 0; s < world; ++s) {
      uint64_t k = g->meta[s][0];
      if (k && cudaMemcpyAsync((char *)recv + recv_off[s] * (size_t)row_bytes, g->ptr[s], k * (size_t)row_bytes, cudaMemcpyDefault, st) != cudaSuccess) return BKID_ERR_CUDA;
    }
    cudaStreamSynchronize(st);
    if (!g->barrier()) { err = "another rank failed"; return BKID_ERR_ARG; }
    return 0;
  }
  int relay_i64(long long *v, int from, int to) override
  {
    if (rank == from) g->relay = *v;
    if (!g->barrier()) { err = "another rank failed"; return BKID_ERR_ARG; }
    if (rank == to) *v = g->relay;
    if (!g->barrier()) { err = "another rank failed"; return BKID_ERR_ARG; }
    return 0;
  }
};

// ---- NCCL (dlopen: the library stays loadable, and single-GPU use stays possible, without it) ----------------------
struct NcclApi {
  void *h = nullptr;
  typedef struct { char internal[128]; } uid_t;
  int (*GetUniqueId)(uid_t *) = nullptr;
  int (*CommInitRank)(void **, int, uid_t, int) = nullptr;
  int (*CommInitAll)(void **, int, const int *) = nullptr;
  int (*CommDestroy)(void *) = nullptr;
  int (*AllReduce)(const void *, void *, size_t, int, int, void *, cudaStream_t) = nullptr;
  int (*AllGather)(const void *, void *, size_t, int, void *, cudaStream_t) = nullptr;
  int (*Send)(const void *, size_t, int, int, void *, cudaStream_t) = nullptr;
  int (*Recv)(void *, size_t, int, int, void *, cudaStream_t) = nullptr;
  int (*GroupStart)() = nullptr;
  int (*GroupEnd)() = nullptr;
  const char *(*GetErrorString)(int) = nullptr;
  bool load(std::string &err)
  {
    if (h) return true;
    for (const char *name : {"libnccl.so.2", "libnccl.so"}) { h = dlopen(name, RTLD_NOW | RTLD_GLOBAL); if (h) break; }
    if (!h) { err = std::string("cannot load libnccl.so.2: ") + (dlerror() ? dlerror() : "?"); return false; }
#define BK_NCCL_SYM(f) *(void **)(&f) = dlsym(h, "nccl" #f); if (!f) { err = "libnccl lacks nccl" #f; return false; }
    BK_NCCL_SYM(GetUniqueId) BK_NCCL_SYM(CommInitRank) BK_NCCL_SYM(CommInitAll) BK_NCCL_SYM(CommDestroy) BK_NCCL_SYM(AllReduce) BK_NCCL_SYM(AllGather)
    BK_NCCL_SYM(Send) BK_NCCL_SYM(Recv) BK_NCCL_SYM(GroupStart) BK_NCCL_SYM(GroupEnd) BK_NCCL_SYM(GetErrorString)
#undef BK_NCCL_SYM
    return true;
  }
};
static NcclApi g_nccl;
enum { NCCL_CHAR = 0, NCCL_UINT32 = 3, NCCL_UINT64 = 5, NCCL_OP_SUM = 0, NCCL_OP_MAX = 2 };   // ncclDataType_t / ncclRedOp_t (nccl.h)

struct NcclComm : bkid_comm {
  void *comm = nullptr;
  int device = 0;
  DBuf scratch;                                               // small device buffer for the host-metadata all-gather
  ~NcclComm() override { if (comm) g_nccl.CommDestroy(comm); scratch.release(); }
  int chk(int rc, const char *what) { if (rc != 0) { err = std::string(what) + ": " + g_nccl.GetErrorString(rc); return BKID_ERR_CUDA; } return 0; }
  int allreduce(void *dev, int n, BkType ty, BkOp op, cudaStream_t st) override
  {
    if (n <= 0) return 0;
    BK_TRY(chk(g_nccl.AllReduce(dev, dev, (size_t)n, ty == BK_U64 ? NCCL_UINT64 : NCCL_UINT32, op == BK_SUM ? NCCL_OP_SUM : NCCL_OP_MAX, comm, st), "ncclAllReduce"));
    return cudaStreamSynchronize(st) == cudaSuccess ? 0 : BKID_ERR_CUDA;
  }
  int allgather_host(const uint64_t *mine, int n, uint64_t *all) override
  {
    cudaStream_t st = nullptr;                                // legacy stream is fine for this tiny metadata exchange
    BK_TRY(scratch.ensure((size_t)(world + 1) * n * 8 + 64, 0, st));
    uint64_t *d = scratch.as<uint64_t>();
    if (cudaMemcpy(d, mine, (size_t)n * 8, cudaMemcpyHostToDevice) != cudaSuccess) return BKID_ERR_CUDA;
    BK_TRY(chk(g_nccl.AllGather(d, d + n, (size_t)n, NCCL_UINT64, comm, st), "ncclAllGather"));
    return cudaMemcpy(all, d + n, (size_t)world * n * 8, cudaMemcpyDeviceToHost) == cudaSuccess ? 0 : BKID_ERR_CUDA;
  }
  int alltoallv(const void *send, const uint64_t *send_off, void *recv, const uint64_t *recv_off, int row_bytes, cudaStream_t st) override
  {
    BK_TRY(chk(g_nccl.GroupStart(), "ncclGroupStart"));
    for (int r = 0; r < world; ++r) {
      uint64_t ns = send_off[r + 1] - send_off[r], nr = recv_off[r + 1] - recv_off[r];
      if (ns) BK_TRY(chk(g_nccl.Send((const char *)send + send_off[r] * (size_t)row_bytes, ns * (size_t)row_bytes, NCCL_CHAR, r, comm, st), "ncclSend"));
      if (nr) BK_TRY(chk(g_nccl.Recv((char *)recv + recv_off[r] * (size_t)row_bytes, nr * (size_t)row_bytes, NCCL_CHAR, r, comm, st), "ncclRecv"));
    }
    BK_TRY(chk(g_nccl.GroupEnd(), "ncclGroupEnd"));
    return cudaStreamSynchronize(st) == cudaSuccess ? 0 : BKID_ERR_CUDA;
  }
  int allgatherv(const void *send, uint64_t nrows, void *recv, const uint64_t *recv_off, int row_bytes, cudaStream_t st) override
  {
    BK_TRY(chk(g_nccl.GroupStart(), "ncclGroupStart"));
    for (int r = 0; r < world; ++r) {
      uint64_t nr = recv_off[r + 1] - recv_off[r];
      if (nrows) BK_TRY(chk(g_nccl.Send(send, nrows * (size_t)row_bytes, NCCL_CHAR, r, comm, st), "ncclSend"));
      if (nr) BK_TRY(chk(g_nccl.Recv((char *)recv + recv_off[r] * (size_t)row_bytes, nr * (size_t)row_bytes, NCCL_CHAR, r, comm, st), "ncclRecv"));
    }
    BK_TRY(chk(g_nccl.GroupEnd(), "ncclGroupEnd"));
    return cudaStreamSynchronize(st) == cudaSuccess ? 0 : BKID_ERR_CUDA;
  }
  int relay_i64(long long *v, int from, int to) override
  {
    if (rank != from && rank != to) return 0;
    cudaStream_t st = nullptr;
    BK_TRY(scratch.ensure(64, 0, st));
    long long *d = scratch.as<long long>();
    if (rank == from) {
      if (cudaMemcpy(d, v, 8, cudaMemcpyHostToDevice) != cudaSuccess) return BKID_ERR_CUDA;
      BK_TRY(chk(g_nccl.Send(d, 8, NCCL_CHAR, to, comm, st), "ncclSend"));
      return cudaStreamSynchronize(st) == cudaSuccess ? 0 : BKID_ERR_CUDA;
    }
    BK_TRY(chk(g_nccl.Recv(d, 8, NCCL_CHAR, from, comm, st), "ncclRecv"));
    return cudaMemcpy(v, d, 8, cudaMemcpyDeviceToHost) == cudaSuccess ? 0 : BKID_ERR_CUDA;
  }
};

// ---------------------------------------------------------------------------------------------------------------
// routing kernels: owner of a row + stable partition by owner (W <= 32), fused
// ---------------------------------------------------------------------------------------------------------------
constexpr int RT_THREADS = 256;
constexpr int RT_MAXW = 32;

// owner of a candidate = f(name hash): both mates of a read meet on one rank without trusting the mate fields
__device__ __forceinline__ uint32_t cand_owner(const bkid_cand &c, uint32_t W) { return (uint32_t)((c.name_lo >> 8) & 0x7fffffffull) % W; }

template <int MODE>   // 0: candidate rows by name hash, 1: pair rows by owner_of_bucket[bucket rank]
__device__ __forceinline__ uint32_t row_owner(const void *rows, long long i, uint32_t W, const uint8_t *__restrict__ table)
{
  if (MODE == 0) return cand_owner(reinterpret_cast<const bkid_cand *>(rows)[i], W);
  return table[reinterpret_cast<const bkid_pair *>(rows)[i].bucket];
}

template <int MODE>
__global__ void __launch_bounds__(RT_THREADS) rt_count(const void *__restrict__ rows, long long n, uint32_t W, const uint8_t *__restrict__ table, uint32_t *__restrict__ tile_cnt /* [W][ntiles] */, int ntiles)
{
  __shared__ unsigned h[RT_MAXW];
  if (threadIdx.x < RT_MAXW) h[threadIdx.x] = 0;
  __syncthreads();
  long long i = (long long)blockIdx.x * RT_THREADS + threadIdx.x;
  unsigned o = i < n ? row_owner<MODE>(rows, i, W, table) : 0xffffffffu;
  unsigned m = __match_any_sync(0xffffffffu, o);
  if (i < n && (threadIdx.x & 31) == (unsigned)(__ffs(m) - 1)) atomicAdd(&h[o], (unsigned)__popc(m));
  __syncthreads();
  if (threadIdx.x < W) tile_cnt[(size_t)threadIdx.x * ntiles + blockIdx.x] = h[threadIdx.x];
}

template <int MODE>
__global__ void __launch_bounds__(RT_THREADS) rt_scatter(const void *__restrict__ rows, long long n, uint32_t W, const uint8_t *__restrict__ table, const uint32_t *__restrict__ tile_off /* [W][ntiles] scanned */,
                                                         int ntiles, int row_chunks /* 16-byte chunks per row */, uint4 *__restrict__ out)
{
  __shared__ unsigned wcnt[RT_THREADS / 32][RT_MAXW];
  const unsigned w = threadIdx.x >> 5, l = threadIdx.x & 31;
  for (int k = threadIdx.x; k < (RT_THREADS / 32) * RT_MAXW; k += RT_THREADS) (&wcnt[0][0])[k] = 0;
  __syncthreads();
  long long i = (long long)blockIdx.x * RT_THREADS + threadIdx.x;
  unsigned o = i < n ? row_owner<MODE>(rows, i, W, table) : 0xffffffffu;
  unsigned m = __match_any_sync(0xffffffffu, o);
  unsigned before = __popc(m & ((1u << l) - 1u));
  if (i < n && before == 0) wcnt[w][o] = (unsigned)__popc(m);
  __syncthreads();
  if (i >= n) return;
  unsigned base = tile_off[(size_t)o * ntiles + blockIdx.x];
  for (unsigned ww = 0; ww < w; ++ww) base += wcnt[ww][o];
  const uint4 *src = reinterpret_cast<const uint4 *>(rows) + i * row_chunks;
  uint4 *dst = out + (size_t)(base + before) * row_chunks;
  for (int k = 0; k < row_chunks; ++k) dst[k] = src[k];
}

__global__ void pair_bucket_hist(const bkid_pair *__restrict__ pairs, long long n, unsigned *__restrict__ hist)
{
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) atomicAdd(&hist[pairs[i].bucket], 1u);
}
__global__ void rows_sorted_check(const bkid_sarow *__restrict__ rows, long long n, int *__restrict__ bad)
{
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i + 1 >= n) return;
  const EvRow &a = reinterpret_cast<const EvRow *>(rows)[i], &b = reinterpret_cast<const EvRow *>(rows)[i + 1];
  uint32_t ta = (uint32_t)a.tid, tb = (uint32_t)b.tid;
  if (ta > tb || (ta == tb && a.pos > b.pos)) atomicExch(bad, 1);
}
__global__ void cluster_bucket_dense(bkid_cluster_rec *cl, uint32_t n, const int32_t *__restrict__ ranks, int nranks)
{
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  int a = 0, b = nranks;                                     // first k with ranks[k] >= bucket rank
  int v = cl[i].bucket;
  while (a < b) { int m = (a + b) >> 1; if (ranks[m] < v) a = m + 1; else b = m; }
  cl[i].bucket = a;
}

// stable partition of n rows by owner: out = rows grouped by owner (each group in input order), send_off[W+1] on the host
template <int MODE>
static int route_rows(bkid_ctx *c, const void *rows, long long n, int row_bytes, uint32_t W, const uint8_t *table, DBuf &out, std::vector<uint64_t> &send_off)
{
  cudaStream_t st = c->st;
  send_off.assign(W + 1, 0);
  TRY(c, out.ensure((size_t)std::max<long long>(n, 1) * row_bytes, 0, st));
  if (n <= 0) return 0;
  int ntiles = div_up(n, RT_THREADS);
  size_t cells = (size_t)W * ntiles;
  TRY(c, c->sc.ensure((long long)cells + 8, st));
  uint32_t *cnt = c->sc.a32.as<uint32_t>(), *off = c->sc.b32.as<uint32_t>();
  BK_LAUNCH((rt_count<MODE>), ntiles, RT_THREADS, 0, st, rows, n, W, table, cnt, ntiles);
  bk::exclusive_scan<uint32_t, uint32_t>(cnt, off, (long long)cells, c->sc.scan_tmp.as<unsigned long long>(), nullptr, st);
  BK_LAUNCH((rt_scatter<MODE>), ntiles, RT_THREADS, 0, st, rows, n, W, table, off, ntiles, row_bytes / 16, out.as<uint4>());
  // group starts = scanned offset of each owner's first tile
  std::vector<uint32_t> h(W);
  for (uint32_t r = 0; r < W; ++r) CU(c, cudaMemcpyAsync(&h[r], off + (size_t)r * ntiles, 4, cudaMemcpyDeviceToHost, st));
  TRY(c, sync_check(c));
  for (uint32_t r = 0; r < W; ++r) send_off[r] = h[r];
  send_off[W] = (uint64_t)n;
  return 0;
}

static int exchange_rows(bkid_ctx *c, bkid_comm *cm, const DBuf &send, const std::vector<uint64_t> &send_off, int row_bytes, DBuf &recv, long long *n_recv)
{
  int W = cm->world;
  std::vector<uint64_t> cnt(W), all((size_t)W * W), recv_off(W + 1, 0);
  for (int r = 0; r < W; ++r) cnt[r] = send_off[r + 1] - send_off[r];
  if (cm->allgather_host(cnt.data(), W, all.data())) return fail(c, BKID_ERR_CUDA, "count exchange failed: " + cm->err);
  for (int s = 0; s < W; ++s) recv_off[s + 1] = recv_off[s] + all[(size_t)s * W + cm->rank];
  TRY(c, recv.ensure((size_t)std::max<uint64_t>(recv_off[W], 1) * row_bytes, 0, c->st));
  if (cm->alltoallv(send.p, send_off.data(), recv.p, recv_off.data(), row_bytes, c->st)) return fail(c, BKID_ERR_CUDA, "all-to-all failed: " + cm->err);
  *n_recv = (long long)recv_off[W];
  return 0;
}

static int gather_rows_all(bkid_ctx *c, bkid_comm *cm, const void *mine, long long n_mine, int row_bytes, DBuf &recv, long long *n_all)
{
  int W = cm->world;
  uint64_t k = (uint64_t)n_mine;
  std::vector<uint64_t> all(W), off(W + 1, 0);
  if (cm->allgather_host(&k, 1, all.data())) return fail(c, BKID_ERR_CUDA, "count exchange failed: " + cm->err);
  for (int s = 0; s < W; ++s) off[s + 1] = off[s] + all[s];
  TRY(c, recv.ensure((size_t)std::max<uint64_t>(off[W], 1) * row_bytes, 0, c->st));
  if (cm->allgatherv(mine, k, recv.p, off.data(), row_bytes, c->st)) return fail(c, BKID_ERR_CUDA, "all-gather failed: " + cm->err);
  *n_all = (long long)off[W];
  return 0;
}

// bucket -> rank by longest-processing-time-first on the GLOBAL pairs-per-bucket histogram (identical on every rank)
static void lpt_owner_table(const std::vector<unsigned long long> &hist, int W, std::vector<uint8_t> &owner)
{
  std::vector<int> order;
  for (int b = 0; b < (int)hist.size(); ++b) if (hist[b]) order.push_back(b);
  std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return hist[a] > hist[b]; });
  std::vector<double> load(W, 0.0);
  owner.assign(hist.size(), 0);
  for (int b : order) {
    int best = 0;
    for (int r = 1; r < W; ++r) if (load[r] < load[best]) best = r;
    owner[b] = (uint8_t)best;
    double m = (double)hist[b];
    load[best] += m * (1.0 + log2(m + 1.0) / 16.0);          // sort replay + clustering grow a little faster than linearly
  }
}

// ---------------------------------------------------------------------------------------------------------------
// the sharded hot path (collective: every rank calls it with its own context)
// ---------------------------------------------------------------------------------------------------------------
struct DistTimes { float stats = 0, candidates = 0, a2a_cand = 0, join = 0, a2a_pairs = 0, cluster = 0, gather = 0, refine = 0, total = 0; };

static int dist_run_impl(bkid_ctx *c, bkid_comm *cm, int mode, double *mean_o, double *sd_o, double *dist_o, int64_t *n_called, DistTimes *tmo)
{
  const int W = cm->world, R = cm->rank;
  cudaSetDevice(c->device);
  c->err.clear();
  cudaStream_t st = c->st;
  auto now = [] { return std::chrono::steady_clock::now(); };
  auto ms_since = [](std::chrono::steady_clock::time_point t0) { return std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t0).count(); };
  auto T0 = now(), t0 = T0;
  DistTimes tm;
  if (W > RT_MAXW) return fail(c, BKID_ERR_ARG, "more than 32 ranks");
  // ---- insert statistics ----
  TRY(c, classify_impl(c));
  TRY(c, c->dist_scalars.ensure(4096, 0, st));
  unsigned long long *dv = c->dist_scalars.as<unsigned long long>();
  unsigned long long hv[4] = {(unsigned long long)c->sum_abs, (unsigned long long)c->cnt_insert, c->sum_sq, (unsigned long long)c->n};
  CU(c, cudaMemcpyAsync(dv, hv, 32, cudaMemcpyHostToDevice, st));
  if (cm->allreduce(dv, 3, BK_U64, BK_SUM, st)) return fail(c, BKID_ERR_CUDA, "all-reduce failed: " + cm->err);
  unsigned long long xm = c->xmax;
  CU(c, cudaMemcpyAsync(dv + 8, &xm, 8, cudaMemcpyHostToDevice, st));
  if (cm->allreduce(dv + 8, 1, BK_U64, BK_MAX, st)) return fail(c, BKID_ERR_CUDA, "all-reduce failed: " + cm->err);
  unsigned long long gs[3], gxm;
  CU(c, cudaMemcpyAsync(gs, dv, 24, cudaMemcpyDeviceToHost, st)); CU(c, cudaMemcpyAsync(&gxm, dv + 8, 8, cudaMemcpyDeviceToHost, st));
  TRY(c, sync_check(c));
  const unsigned long long N = gs[1];
  TRY(c, stats_begin(c, gs[0], N, gs[2], gxm, c->st2));                       // one streaming pass on every rank at once, on the side stream
  // global index of my first record
  std::vector<uint64_t> ns(W);
  { uint64_t mine = (uint64_t)c->n; if (cm->allgather_host(&mine, 1, ns.data())) return fail(c, BKID_ERR_CUDA, "count exchange failed: " + cm->err); }
  unsigned long long offset = 0;
  for (int r = 0; r < R; ++r) offset += ns[r];
  tm.stats = ms_since(t0); t0 = now();
  // ---- candidates meet their mates on the owner of their name hash ----
  TRY(c, extract_candidates(c, offset, false));
  {
    unsigned hnc[2] = {0, 0};
    CU(c, cudaMemcpyAsync(hnc, c->counters.as<unsigned>() + CS_NC, 8, cudaMemcpyDeviceToHost, st));
    TRY(c, sync_check(c));
    TRY(c, check_candidates(c, hnc));
  }
  tm.candidates = ms_since(t0); t0 = now();
  std::vector<uint64_t> soff;
  TRY(c, route_rows<0>(c, c->cand.p, c->n_cand, (int)sizeof(bkid_cand), (uint32_t)W, nullptr, c->dist_send, soff));
  long long nc_all = 0;
  TRY(c, exchange_rows(c, cm, c->dist_send, soff, (int)sizeof(bkid_cand), c->dist_recv, &nc_all));
  tm.a2a_cand = ms_since(t0); t0 = now();
  // ---- sd: exact and order independent when no record can need a correction ----
  unsigned long long fe[2] = {0, 0};
  TRY(c, stats_collect(c, &fe[0], &fe[1]));
  CU(c, cudaMemcpyAsync(dv + 16, fe, 16, cudaMemcpyHostToDevice, st));
  if (cm->allreduce(dv + 16, 2, BK_U64, BK_SUM, st)) return fail(c, BKID_ERR_CUDA, "all-reduce failed: " + cm->err);
  CU(c, cudaMemcpyAsync(fe, dv + 16, 16, cudaMemcpyDeviceToHost, st));
  TRY(c, sync_check(c));
  long long total = (long long)fe[0];
  if (fe[1] != 0) {                                                            // the order-dependent replay, chained through the ranks
    TRY(c, stats_prepare(c, c->mean));
    long long t = 0;
    for (int src = 0; src < W; ++src) {
      if (R == src) TRY(c, stats_replay(c, c->mean, t, &t));
      if (src + 1 < W && cm->relay_i64(&t, src, src + 1)) return fail(c, BKID_ERR_CUDA, "sd relay failed: " + cm->err);
    }
    // the last rank holds the total: everybody gets it
    unsigned long long tv = R == W - 1 ? (unsigned long long)t : 0ull;
    CU(c, cudaMemcpyAsync(dv + 24, &tv, 8, cudaMemcpyHostToDevice, st));
    if (cm->allreduce(dv + 24, 1, BK_U64, BK_SUM, st)) return fail(c, BKID_ERR_CUDA, "all-reduce failed: " + cm->err);
    CU(c, cudaMemcpyAsync(&tv, dv + 24, 8, cudaMemcpyDeviceToHost, st));
    TRY(c, sync_check(c));
    total = (long long)tv;
  }
  stats_set(c, total, (long long)N);
  const int times = c->prm.times;
  const double d = times * sqrt((double)times) * (c->mean + c->prm.sd_mult * c->sd); // :103
  // ---- join (the received candidates are in global file order: sources in rank order, each in its own order) ----
  long long np = 0;
  TRY(c, join_candidates(c, c->dist_recv.as<bkid_cand>(), nc_all, d, &np));
  tm.join = ms_since(t0); t0 = now();
  // ---- pairs go to the owner of their chr-pair bucket: LPT on the global bucket histogram ----
  const int nbk = (c->nt + 1) * (c->nt + 1);
  TRY(c, c->tmpF.ensure((size_t)nbk * 8 + 64, 0, st));
  unsigned *bh = c->tmpF.as<unsigned>();
  CU(c, cudaMemsetAsync(bh, 0, (size_t)nbk * 4, st));
  if (np > 0) BK_LAUNCH(pair_bucket_hist, GRID1(np, 256), 256, 0, st, c->pairs_tmp.as<bkid_pair>(), np, bh);
  if (cm->allreduce(bh, nbk, BK_U32, BK_SUM, st)) return fail(c, BKID_ERR_CUDA, "all-reduce failed: " + cm->err);
  std::vector<unsigned> hb(nbk);
  CU(c, cudaMemcpyAsync(hb.data(), bh, (size_t)nbk * 4, cudaMemcpyDeviceToHost, st));
  TRY(c, sync_check(c));
  std::vector<unsigned long long> hist(hb.begin(), hb.end());
  std::vector<uint8_t> owner;
  lpt_owner_table(hist, W, owner);
  uint8_t *d_owner = (uint8_t *)(bh + nbk);
  CU(c, cudaMemcpyAsync(d_owner, owner.data(), (size_t)nbk, cudaMemcpyHostToDevice, st));
  TRY(c, route_rows<1>(c, c->pairs_tmp.p, np, (int)sizeof(bkid_pair), (uint32_t)W, d_owner, c->dist_send, soff));
  long long np_all = 0;
  TRY(c, exchange_rows(c, cm, c->dist_send, soff, (int)sizeof(bkid_pair), c->dist_recv, &np_all));
  tm.a2a_pairs = ms_since(t0); t0 = now();
  TRY(c, set_pairs(c, c->dist_recv.as<bkid_pair>(), np_all, false));
  c->tm.n_pairs = c->np0;
  c->scanned = true; c->clustered = c->refined = false;
  int64_t ncl_local = 0;
  TRY(c, bkid_cluster(c, d, mode, &ncl_local));
  tm.cluster = ms_since(t0); t0 = now();
  // ---- every rank gets every cluster summary, in the reference's order (bucket name rank, cluster id) ----
  const bkid_cluster_rec *cl_dev = nullptr; int64_t ncl_mine = 0;
  TRY(c, bkid_shard_clusters(c, &cl_dev, &ncl_mine));
  long long ncl_all = 0;
  TRY(c, gather_rows_all(c, cm, cl_dev, ncl_mine, (int)sizeof(bkid_cluster_rec), c->dist_recv, &ncl_all));
  {
    std::vector<bkid_cluster_rec> hcl((size_t)std::max<long long>(ncl_all, 1));
    if (ncl_all) CU(c, cudaMemcpyAsync(hcl.data(), c->dist_recv.p, (size_t)ncl_all * sizeof(bkid_cluster_rec), cudaMemcpyDeviceToHost, st));
    TRY(c, sync_check(c));
    hcl.resize((size_t)ncl_all);
    std::stable_sort(hcl.begin(), hcl.end(), [](const bkid_cluster_rec &a, const bkid_cluster_rec &b) { return a.bucket != b.bucket ? a.bucket < b.bucket : a.id < b.id; });
    TRY(c, c->clusters.ensure((size_t)(ncl_all + 1) * sizeof(bkid_cluster_rec), 0, st));
    if (ncl_all) CU(c, cudaMemcpyAsync(c->clusters.p, hcl.data(), (size_t)ncl_all * sizeof(bkid_cluster_rec), cudaMemcpyHostToDevice, st));
    TRY(c, sync_check(c));
    c->n_clusters = ncl_all; c->clusters_ranked = true; c->clustered = true; c->refined = false;
  }
  // bucket name ranks that hold at least one pair, over all ranks (the reference's dense bucket ids)
  std::vector<int32_t> all_ranks;
  {
    int64_t nbl = c->nb;
    long long nb_all = 0;
    TRY(c, gather_rows_all(c, cm, c->bucket_rank_of.p, nbl, 4, c->dist_send, &nb_all));
    all_ranks.resize((size_t)nb_all);
    if (nb_all) CU(c, cudaMemcpyAsync(all_ranks.data(), c->dist_send.p, (size_t)nb_all * 4, cudaMemcpyDeviceToHost, st));
    TRY(c, sync_check(c));
    std::sort(all_ranks.begin(), all_ranks.end());
  }
  // ---- split-read evidence rows of all ranks (coordinate order = rank order) ----
  TRY(c, refine_build_rows(c));
  long long nrows_all = 0;
  TRY(c, gather_rows_all(c, cm, c->sarows.p, c->n_sa, (int)sizeof(bkid_sarow), c->dist_rows, &nrows_all));
  {
    int *bad = (int *)(c->counters.as<unsigned>() + CS_MISSING);
    CU(c, cudaMemsetAsync(bad, 0, 4, st));
    if (nrows_all > 1) BK_LAUNCH(rows_sorted_check, GRID1(nrows_all, 256), 256, 0, st, (const bkid_sarow *)c->dist_rows.p, nrows_all, bad);
    int hbad = 0;
    CU(c, cudaMemcpyAsync(&hbad, bad, 4, cudaMemcpyDeviceToHost, st));
    TRY(c, sync_check(c));
    if (hbad) return fail(c, BKID_ERR_ARG, "the ranks' record slices are not in coordinate order (rank r must hold the r-th genomic bin)");
  }
  c->rows_ptr = c->dist_rows.p; c->n_rows = nrows_all;
  tm.gather = ms_since(t0); t0 = now();
  // ---- refinement: partial region coverage / depth per shard, summed over the ranks ----
  c->n_called = 0;
  if (ncl_all > 0) {
    int ms_local = 0;
    TRY(c, refine_local_maxspan(c, &ms_local));
    unsigned long long msv = (unsigned long long)ms_local;
    CU(c, cudaMemcpyAsync(dv + 32, &msv, 8, cudaMemcpyHostToDevice, st));
    if (cm->allreduce(dv + 32, 1, BK_U64, BK_MAX, st)) return fail(c, BKID_ERR_CUDA, "all-reduce failed: " + cm->err);
    CU(c, cudaMemcpyAsync(&msv, dv + 32, 8, cudaMemcpyDeviceToHost, st));
    TRY(c, sync_check(c));
    c->maxspan = (int)msv;
    TRY(c, refine_coverage(c, d));
    if (cm->allreduce(c->cov.p, (int)(2 * ncl_all), BK_U32, BK_SUM, st)) return fail(c, BKID_ERR_CUDA, "all-reduce failed: " + cm->err);
    TRY(c, refine_vote(c));
    TRY(c, refine_depth(c));
    if (cm->allreduce(c->depth.p, (int)(2 * ncl_all), BK_U32, BK_SUM, st)) return fail(c, BKID_ERR_CUDA, "all-reduce failed: " + cm->err);
    TRY(c, refine_finish(c));
    if (c->n_called > 0 && !all_ranks.empty()) {                               // bucket name rank -> dense bucket id
      TRY(c, c->tmpF.ensure(all_ranks.size() * 4 + 64, 0, st));
      CU(c, cudaMemcpyAsync(c->tmpF.p, all_ranks.data(), all_ranks.size() * 4, cudaMemcpyHostToDevice, st));
      BK_LAUNCH(cluster_bucket_dense, GRID1(c->n_called, 128), 128, 0, st, c->clusters_out.as<bkid_cluster_rec>(), (uint32_t)c->n_called, c->tmpF.as<int32_t>(), (int)all_ranks.size());
      TRY(c, sync_check(c));
    }
  } else {
    // keep the collective call sequence identical on every rank: nothing to do when there is no cluster anywhere
  }
  c->refined = true;
  c->tm.n_called = c->n_called;
  tm.refine = ms_since(t0);
  tm.total = ms_since(T0);
  if (mean_o) *mean_o = c->mean;
  if (sd_o) *sd_o = c->sd;
  if (dist_o) *dist_o = d;
  if (n_called) *n_called = c->n_called;
  if (tmo) *tmo = tm;
  return 0;
}

extern "C" {

bkid_comm *bkid_comm_nccl_init(const uint8_t *unique_id /* 128 bytes from rank 0 */, int rank, int world, int device)
{
  std::string err;
  if (!g_nccl.load(err)) { g_create_err = err; return nullptr; }
  if (cudaSetDevice(device) != cudaSuccess) { g_create_err = "cudaSetDevice failed"; return nullptr; }
  NcclComm *cm = new NcclComm();
  cm->rank = rank; cm->world = world; cm->device = device;
  NcclApi::uid_t id;
  memcpy(&id, unique_id, sizeof id);
  int rc = g_nccl.CommInitRank(&cm->comm, world, id, rank);
  if (rc != 0) { g_create_err = std::string("ncclCommInitRank: ") + g_nccl.GetErrorString(rc); cm->comm = nullptr; delete cm; return nullptr; }
  return cm;
}

int bkid_comm_nccl_unique_id(uint8_t *out /* 128 bytes */)
{
  std::string err;
  if (!g_nccl.load(err)) { g_create_err = err; return BKID_ERR_CUDA; }
  NcclApi::uid_t id;
  int rc = g_nccl.GetUniqueId(&id);
  if (rc != 0) { g_create_err = std::string("ncclGetUniqueId: ") + g_nccl.GetErrorString(rc); return BKID_ERR_CUDA; }
  memcpy(out, &id, sizeof id);
  return 0;
}

// one communicator per device of ONE process (ranks = host threads): the BreakID driver with -gpu 0,1,...
int bkid_comm_nccl_init_all(const int *devices, int world, bkid_comm **out)
{
  std::string err;
  if (!g_nccl.load(err)) { g_create_err = err; return BKID_ERR_CUDA; }
  std::vector<void *> comms(world, nullptr);
  int rc = g_nccl.CommInitAll(comms.data(), world, devices);
  if (rc != 0) { g_create_err = std::string("ncclCommInitAll: ") + g_nccl.GetErrorString(rc); return BKID_ERR_CUDA; }
  for (int r = 0; r < world; ++r) { NcclComm *cm = new NcclComm(); cm->rank = r; cm->world = world; cm->device = devices[r]; cm->comm = comms[r]; out[r] = cm; }
  return 0;
}

// ranks = host threads of this process, exchanges = device copies behind a barrier (contexts may share a device)
int bkid_comm_local_create(int world, bkid_comm **out)
{
  if (world < 1 || !out) return BKID_ERR_ARG;
  auto grp = std::make_shared<LocalGroup>(world);
  for (int r = 0; r < world; ++r) out[r] = new LocalComm(grp, r);
  return 0;
}

void bkid_comm_destroy(bkid_comm *cm) { delete cm; }

// the bucket -> rank table bkid_dist_run derives from the global pairs-per-bucket histogram (pure host code; exported so
// that the CPU test-suite can check it: every rank must compute the same table from the same histogram)
int bkid_lpt_owner_table(const uint64_t *hist, int n_buckets, int world, uint8_t *owner)
{
  if (!hist || !owner || n_buckets < 0 || world < 1 || world > RT_MAXW) return BKID_ERR_ARG;
  std::vector<unsigned long long> h(hist, hist + n_buckets);
  std::vector<uint8_t> o;
  lpt_owner_table(h, world, o);
  if (n_buckets) memcpy(owner, o.data(), (size_t)n_buckets);
  return 0;
}

int bkid_dist_run(bkid_ctx *c, bkid_comm *cm, int mode, double *mean, double *sd, double *dist, int64_t *n_called, float *stage_ms /* [9] or NULL */)
{
  if (!c || !cm) return BKID_ERR_ARG;
  DistTimes tm;
  int rc = dist_run_impl(c, cm, mode, mean, sd, dist, n_called, &tm);
  if (rc) cm->abort();
  if (stage_ms) { float v[9] = {tm.stats, tm.candidates, tm.a2a_cand, tm.join, tm.a2a_pairs, tm.cluster, tm.gather, tm.refine, tm.total}; memcpy(stage_ms, v, sizeof v); }
  return rc;
}

// the same with one host thread per rank (contexts and communicators of this process): returns the first failure
int bkid_dist_run_threads(bkid_ctx **ctxs, bkid_comm **comms, int world, int mode, double *mean, double *sd, double *dist, int64_t *n_called)
{
  if (!ctxs || !comms || world < 1) return BKID_ERR_ARG;
  std::vector<int> rcs(world, 0);
  std::vector<std::thread> th;
  for (int r = 0; r < world; ++r)
    th.emplace_back([&, r] {
      rcs[r] = dist_run_impl(ctxs[r], comms[r], mode, mean ? mean + r : nullptr, sd ? sd + r : nullptr, dist ? dist + r : nullptr, n_called ? n_called + r : nullptr, nullptr);
      if (rcs[r]) comms[r]->abort();
    });
  for (auto &t : th) t.join();
  for (int r = 0; r < world; ++r) if (rcs[r]) return rcs[r];
  return 0;
}

}  // extern "C"
