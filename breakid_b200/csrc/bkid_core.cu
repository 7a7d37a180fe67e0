// bkid_core.cu -- CUDA (sm_100a) implementation of BreakID's data-parallel core behind the C ABI of
// include/breakid_b200.h.  Written from scratch for B200: every stage is HBM-bound integer / FP64
// scalar work (no dense contraction anywhere on this path, so no tensor cores), laid out as
// struct-of-arrays columns resident in HBM, 128-bit vector loads on the streaming kernels, grids
// sized from the tile count, and no host round trips inside a stage except the small counters a
// stage boundary needs.
//
// Reference files cited below are relative to the reference tree (SinOncology/BreakID).
//
//   K1  classify + insert statistics        src/BreakID.cc:1419-1420, 1909-1954, util_bed.cc:183
//   K1s exact replay of the truncating sd accumulator (src/BreakID.cc:1913,1944)
//   K2  mate join (radix sort on name hash + pairwise protocol)      src/BreakID.cc:1424-1494
//   K3  bucket ordering + std::sort replay (parallel introsort)      src/BreakID.cc:1274-1282,1500-1512
//   K4  isolated-pair mask                                           src/BreakID.cc:1813-1877
//   K5a AHC by components (closed-form tie rule)                     src/util_cluster.cc:7-396
//   K5b -fast anchored-window sweep                                  src/BreakID.cc:1046-1160
//   K6  cluster summary + 2w filter                                  src/BreakID.cc:297-352
//   K7  split-read evidence (CIGAR / SA arithmetic)                  src/BreakID.cc:868-1037
//   K8  breakpoint vote                                              src/BreakID.cc:577-857
//   K9  depth / AF / type                                            src/util_bed.cc:154-192
//   K10 nib 41-mer + homopolymer                                     src/util_bam.cc:78-122
#include "../../include/breakid_b200.h"
#include "prims.cuh"

#include <algorithm>
#include <array>
#include <cmath>
#include <cstdio>
#include <chrono>
#include <cstring>
#include <memory>
#include <map>
#include <string>
#include <vector>

thread_local long long g_bk_launches = 0;
static thread_local std::string g_last_cuda_err;
static std::string g_create_err;

// ---- per-kernel timing (bkid_profile_kernels / bkid_profile_report) ----------------------------------------------
bool g_bk_prof_on = false;
namespace {
struct ProfRec { const char *name; cudaEvent_t e0, e1; };
std::vector<ProfRec> g_prof_recs;
std::vector<cudaEvent_t> g_prof_pool;
cudaEvent_t prof_event()
{
  if (!g_prof_pool.empty()) { cudaEvent_t e = g_prof_pool.back(); g_prof_pool.pop_back(); return e; }
  cudaEvent_t e; cudaEventCreate(&e); return e;
}
}  // namespace
void bk_prof_begin(const char *name, cudaStream_t st)
{
  ProfRec r{name, prof_event(), prof_event()};
  cudaEventRecord(r.e0, st);
  g_prof_recs.push_back(r);
}
void bk_prof_end(cudaStream_t st) { if (!g_prof_recs.empty()) cudaEventRecord(g_prof_recs.back().e1, st); }

void bk_set_cuda_error(cudaError_t e, const char *file, int line)
{
  char buf[256];
  snprintf(buf, sizeof buf, "CUDA error %d (%s) at %s:%d", (int)e, cudaGetErrorString(e), file, line);
  g_last_cuda_err = buf;
}

using bk::div_up;

enum { F_PAIRED = 0x1, F_PROPER = 0x2, F_UNMAP = 0x4, F_REVERSE = 0x10, F_SECONDARY = 0x100, F_QCFAIL = 0x200, F_DUP = 0x400 };
enum { CL_INSERT = 1, CL_CAND = 2, CL_DEPTH = 4, CL_SPLITOK = 8, CL_EXCL = 16 /* record lies in an exclude interval: invisible to every stage */ };

// ---------------------------------------------------------------------------------------------
// growable device buffer
// ---------------------------------------------------------------------------------------------
struct DBuf {
  void *p = nullptr;
  size_t cap = 0;
  template <typename T> T *as() const { return (T *)p; }
  // grow to at least `bytes`; keep the first `keep` bytes
  int ensure(size_t bytes, size_t keep, cudaStream_t st)
  {
    if (bytes <= cap) return 0;
    size_t ncap = std::max(bytes, cap + cap / 2);
    ncap = (ncap + 255) & ~(size_t)255;
    void *q = nullptr;
    cudaError_t e = cudaMalloc(&q, ncap);
    if (e != cudaSuccess) { bk_set_cuda_error(e, __FILE__, __LINE__); return e == cudaErrorMemoryAllocation ? BKID_ERR_NOMEM : BKID_ERR_CUDA; }
    if (p && keep) cudaMemcpyAsync(q, p, keep, cudaMemcpyDeviceToDevice, st);
    if (p) { cudaStreamSynchronize(st); cudaFree(p); }
    p = q; cap = ncap;
    return 0;
  }
  void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
};

#define BK_TRY(x) do { int rc__ = (x); if (rc__ != 0) return rc__; } while (0)

// =============================================================================================
// K1: classify + insert statistics (+ maximal reference span).  One block per tile of 4096 records; a
// thread handles 2 groups of 8 consecutive records with 128/64-bit loads and one 64-bit store of the
// class bytes.  The insert-size and span columns come in their narrow forms when the batch has them
// (include/breakid_b200.h: isize16 / span16 -- they stay narrow in HBM):
//   narrow: flag 2 + mapq 1 + isize16 2 + span16 2 read, class 1 written = 8 B/record, max span included
//   wide  : flag 2 + mapq 1 + isize 4 read, class 1 written = 8 B/record (max span: separate pass over pos/endpos)
// Global results g[]: [0] sum |isize|, [1] count, [2] sum isize^2 (all over records passing :1932),
// [3] number of discordant-scan candidates, [4] max |isize| of an insert record, [5] max span.
// =============================================================================================
constexpr int K1_THREADS = 256;
constexpr int K1_TILE = 4096;
enum { G_SUM = 0, G_CNT = 1, G_SQ = 2, G_CAND = 3, G_XMAX = 4, G_SPAN = 5 };

__device__ __forceinline__ unsigned classify_one(unsigned flag, unsigned mapq, int qual)
{
  unsigned c = 0;
  if ((flag & F_PAIRED) && (flag & F_PROPER) && !(flag & (F_UNMAP | F_SECONDARY | F_QCFAIL | F_DUP))) c |= CL_INSERT;      // :1932
  if ((int)mapq >= qual && !(flag & F_DUP) && !(flag & F_SECONDARY) && (flag & F_PAIRED) && !(flag & F_PROPER)) c |= CL_CAND; // :1419-1420
  if (mapq > 0 && !(flag & F_DUP) && (flag & F_PAIRED)) c |= CL_DEPTH;                                                       // util_bed.cc:183
  if (!(flag & F_DUP) && (flag & F_PAIRED)) c |= CL_SPLITOK;                                                                // :898
  return c;
}

// the insert-size column in either form (only records passing :1932 ever read it)
struct ISizeCol {
  const int32_t *w; const int16_t *h;
  __device__ __forceinline__ int at(long long i) const { return h ? (int)h[i] : w[i]; }
};

// four records: packed flag predicates (2 x 16 bit per word), packed mapq predicates (4 x 8 bit)
__device__ __forceinline__ unsigned classify4(unsigned f01, unsigned f23, unsigned m4, unsigned q4, bool q_never, unsigned &ins8)
{
  unsigned ins_lo = __vcmpeq2(f01 & 0x07070707u, 0x00030003u), ins_hi = __vcmpeq2(f23 & 0x07070707u, 0x00030003u);     // :1932
  unsigned bas_lo = __vcmpeq2(f01 & 0x04010401u, 0x00010001u), bas_hi = __vcmpeq2(f23 & 0x04010401u, 0x00010001u);     // !DUP && PAIRED
  unsigned cnd_lo = __vcmpeq2(f01 & 0x05030503u, 0x00010001u), cnd_hi = __vcmpeq2(f23 & 0x05030503u, 0x00010001u);     // :1419-1420 flag part
  ins8 = __byte_perm(ins_lo, ins_hi, 0x6420);
  unsigned bas8 = __byte_perm(bas_lo, bas_hi, 0x6420), cnd8 = __byte_perm(cnd_lo, cnd_hi, 0x6420);
  unsigned ge8 = q_never ? 0u : __vcmpgeu4(m4, q4), gt8 = __vcmpne4(m4, 0u);
  cnd8 &= ge8;
  return (ins8 & 0x01010101u) | (cnd8 & 0x02020202u) | (bas8 & gt8 & 0x04040404u) | (bas8 & 0x08080808u);
}

template <bool I16, bool S16>
__global__ void __launch_bounds__(K1_THREADS)
k1_classify(const uint16_t *__restrict__ flag, const uint8_t *__restrict__ mapq, const int32_t *__restrict__ isize, const int16_t *__restrict__ isize16,
            const uint16_t *__restrict__ span16, long long n, int qual, uint8_t *__restrict__ cls, uint8_t *__restrict__ cand_bits /* [n/8]: bit k of byte i = record 8i+k is a candidate */,
            unsigned long long *__restrict__ g)
{
  __shared__ unsigned long long sh_sum, sh_sq, sh_cnt, sh_cand;
  __shared__ unsigned sh_xmax, sh_span;
  if (threadIdx.x == 0) { sh_sum = 0; sh_sq = 0; sh_cnt = 0; sh_cand = 0; sh_xmax = 0; sh_span = 0; }
  __syncthreads();
  // persistent grid (a few CTAs per SM walk the tiles): the six global results cost one atomic per CTA, not per tile --
  // 150 k tiles x 6 same-sector atomics serialised in L2 and made the kernel 2.4x slower than its memory time
  unsigned long long sum_abs = 0, sum_sq = 0;
  unsigned long long cnt_ins = 0, cnt_cand = 0;
  unsigned xmax = 0, smax2 = 0;
  const unsigned q4 = (unsigned)(qual < 0 ? 0 : (qual > 255 ? 255 : qual)) * 0x01010101u;
  const bool q_never = qual > 255;           // mapq is 8 bits: nothing can pass
  const long long ntiles = (n + K1_TILE - 1) / K1_TILE;
  for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
  const long long tile0 = tile * K1_TILE;
  unsigned cnt = 0;
#pragma unroll
  for (int gq = 0; gq < 2; ++gq) {
    long long i = tile0 + gq * (K1_THREADS * 8) + threadIdx.x * 8;
    if (i + 7 < n) {
      uint4 f8 = *reinterpret_cast<const uint4 *>(flag + i);
      uint2 m8 = *reinterpret_cast<const uint2 *>(mapq + i);
      unsigned insA, insB;
      unsigned cA = classify4(f8.x, f8.y, m8.x, q4, q_never, insA), cB = classify4(f8.z, f8.w, m8.y, q4, q_never, insB);
      *reinterpret_cast<uint2 *>(cls + i) = make_uint2(cA, cB);
      {  // candidate bit of byte k (0x02) -> bit k of one byte: the sparse-table pass reads 1 bit per entry instead of 1 byte
        unsigned a = (cA >> 1) & 0x01010101u, b = (cB >> 1) & 0x01010101u;
        a = (a | (a >> 7) | (a >> 14) | (a >> 21)) & 0xfu; b = (b | (b >> 7) | (b >> 14) | (b >> 21)) & 0xfu;
        cand_bits[i >> 3] = (uint8_t)(a | (b << 4));
      }
      cnt += __popc(cA & 0x01010101u) + __popc(cB & 0x01010101u) + ((__popc(cA & 0x02020202u) + __popc(cB & 0x02020202u)) << 16);
      if (S16) {
        uint4 p8 = *reinterpret_cast<const uint4 *>(span16 + i);
        smax2 = __vmaxu2(__vmaxu2(smax2, p8.x), __vmaxu2(__vmaxu2(p8.y, p8.z), p8.w));
      }
      if (I16) {
        uint4 s8 = *reinterpret_cast<const uint4 *>(isize16 + i);
        // insert masks back to 2 x 16 bit: byte k of ins8 = record k
        unsigned w[4] = {s8.x, s8.y, s8.z, s8.w};
        unsigned mk[4] = {__byte_perm(insA, 0, 0x1100), __byte_perm(insA, 0, 0x3322), __byte_perm(insB, 0, 0x1100), __byte_perm(insB, 0, 0x3322)};
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          unsigned a2 = __vabs2(w[q]) & mk[q];                  // |x| per halfword (|-32768| = 32768 as unsigned), 0 where not an insert record
          unsigned lo = a2 & 0xffffu, hi = a2 >> 16;
          sum_abs += lo + hi;
          sum_sq += (unsigned long long)lo * lo + (unsigned long long)hi * hi;
          xmax = max(xmax, max(lo, hi));
        }
      } else {
        int4 sA = *reinterpret_cast<const int4 *>(isize + i), sB = *reinterpret_cast<const int4 *>(isize + i + 4);
        int sv[8] = {sA.x, sA.y, sA.z, sA.w, sB.x, sB.y, sB.z, sB.w};
#pragma unroll
        for (int q = 0; q < 8; ++q) {
          unsigned mk = (unsigned)((int)(((q < 4 ? insA : insB) << (24 - 8 * (q & 3)))) >> 31);
          unsigned a = (unsigned)(sv[q] < 0 ? -sv[q] : sv[q]) & mk;
          sum_abs += a; sum_sq += (unsigned long long)a * a; xmax = max(xmax, a);
        }
      }
    } else {
      unsigned tail_bits = 0;
      for (int k = 0; k < 8; ++k)
        if (i + k < n) {
          unsigned c = classify_one(flag[i + k], mapq[i + k], qual);
          if (c & CL_INSERT) {
            int sv = I16 ? (int)isize16[i + k] : isize[i + k];
            unsigned a = (unsigned)(sv < 0 ? -sv : sv);
            sum_abs += a; sum_sq += (unsigned long long)a * a; xmax = max(xmax, a); cnt += 1u;
          }
          if (S16) smax2 = __vmaxu2(smax2, (unsigned)span16[i + k]);
          cnt += ((c >> 1) & 1u) << 16;
          cls[i + k] = (uint8_t)c;
          tail_bits |= ((c >> 1) & 1u) << k;
        }
      if (i < n) cand_bits[i >> 3] = (uint8_t)tail_bits;
    }
  }
  cnt_ins += cnt & 0xffffu; cnt_cand += cnt >> 16;      // per tile and thread <= 16 each: the packed counter cannot carry
  }
  unsigned smax = max(smax2 & 0xffffu, smax2 >> 16);
  cnt_ins = bk::warp_sum(cnt_ins); cnt_cand = bk::warp_sum(cnt_cand);
  sum_abs = bk::warp_sum(sum_abs);
  sum_sq = bk::warp_sum(sum_sq);
  for (int o = 16; o; o >>= 1) { xmax = max(xmax, __shfl_xor_sync(0xffffffffu, xmax, o)); smax = max(smax, __shfl_xor_sync(0xffffffffu, smax, o)); }
  if ((threadIdx.x & 31) == 0) { atomicAdd(&sh_cnt, cnt_ins); atomicAdd(&sh_cand, cnt_cand); atomicAdd(&sh_sum, sum_abs); atomicAdd(&sh_sq, sum_sq); atomicMax(&sh_xmax, xmax); atomicMax(&sh_span, smax); }
  __syncthreads();
  if (threadIdx.x == 0) {
    if (sh_cnt) { atomicAdd(g + G_SUM, sh_sum); atomicAdd(g + G_CNT, sh_cnt); atomicAdd(g + G_SQ, sh_sq); atomicMax(g + G_XMAX, (unsigned long long)sh_xmax); }
    if (sh_cand) atomicAdd(g + G_CAND, sh_cand);
    if (S16 && sh_span) atomicMax(g + G_SPAN, (unsigned long long)sh_span);
  }
}

// ---- exclude intervals (extension: north_star's exclude-BED; the reference has no such filter) -----------------
// Semantics: the reference run on a BAM from which every record whose leftmost coordinate (tid, pos) lies in an
// interval has been removed.  Records are coordinate sorted, so an interval is one contiguous record-index range:
// ex_ranges finds it with two binary searches; ex_apply then takes the excluded records back out of what K1
// produced (class byte, insert sum / count, per-tile candidate counts).  K1 itself is untouched and pays nothing.
__device__ __forceinline__ long long ex_lower_bound(const int32_t *__restrict__ tid, const int32_t *__restrict__ pos, long long n, int qt, long long qp)
{
  long long lo = 0, hi = n;
  while (lo < hi) {
    long long m = (lo + hi) >> 1;
    uint32_t tm = (uint32_t)tid[m];
    bool less = tm < (uint32_t)qt || (tm == (uint32_t)qt && (long long)pos[m] < qp);
    if (less) lo = m + 1; else hi = m;
  }
  return lo;
}
// one thread per (merged, sorted) interval; a single trailing thread turns the lengths into a prefix sum
__global__ void ex_ranges(const int32_t *__restrict__ tid, const int32_t *__restrict__ pos, long long n, const int32_t *__restrict__ iv /* [n_iv][3] */, int n_iv,
                          uint32_t *__restrict__ lo, uint32_t *__restrict__ len)
{
  int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n_iv) return;
  long long a = ex_lower_bound(tid, pos, n, iv[3 * k], iv[3 * k + 1]);
  long long b = ex_lower_bound(tid, pos, n, iv[3 * k], iv[3 * k + 2]);
  lo[k] = (uint32_t)a; len[k] = (uint32_t)(b > a ? b - a : 0);
}
__global__ void ex_prefix(const uint32_t *__restrict__ len, int n_iv, unsigned long long *__restrict__ pre /* [n_iv+1] */)
{
  if (blockIdx.x || threadIdx.x) return;
  unsigned long long s = 0;
  for (int k = 0; k < n_iv; ++k) { pre[k] = s; s += len[k]; }
  pre[n_iv] = s;
}
__global__ void __launch_bounds__(256)
ex_apply(const uint32_t *__restrict__ lo, const unsigned long long *__restrict__ pre, int n_iv, ISizeCol isz, uint8_t *__restrict__ cls, uint8_t *__restrict__ cand_bits,
         unsigned long long *__restrict__ g)
{
  unsigned long long E = pre[n_iv];
  unsigned long long sum = 0, sq = 0; unsigned cnt = 0, ncand = 0;
  for (unsigned long long e = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; e < E; e += (unsigned long long)gridDim.x * blockDim.x) {
    int a = 0, b = n_iv;                       // last k with pre[k] <= e
    while (b - a > 1) { int m = (a + b) >> 1; if (pre[m] <= e) a = m; else b = m; }
    long long i = (long long)lo[a] + (long long)(e - pre[a]);
    unsigned c = cls[i];
    if (c & CL_INSERT) { int s = isz.at(i); unsigned long long x = (unsigned long long)(s < 0 ? -(long long)s : (long long)s); sum += x; sq += x * x; ++cnt; }
    if (c & CL_CAND) { ++ncand; atomicAnd(reinterpret_cast<unsigned *>(cand_bits + ((i >> 3) & ~3ll)), ~(1u << (unsigned)(((i >> 3) & 3ll) * 8 + (i & 7)))); }
    cls[i] = (uint8_t)CL_EXCL;
  }
  sum = bk::warp_sum(sum); sq = bk::warp_sum(sq); cnt = bk::warp_sum(cnt); ncand = bk::warp_sum(ncand);
  if ((threadIdx.x & 31) == 0) {
    if (cnt) { atomicAdd(g + G_SUM, 0ull - sum); atomicAdd(g + G_CNT, 0ull - (unsigned long long)cnt); atomicAdd(g + G_SQ, 0ull - sq); }
    if (ncand) atomicAdd(g + G_CAND, 0ull - (unsigned long long)ncand);
  }
}

// =============================================================================================
// K1s: exact replay of `long sd_total += d*d` (src/BreakID.cc:1913,1944).
// The reference converts the long accumulator to double, adds d*d, and truncates back on every
// element: t' = floor(RN(t + a)).  For t + a < 2^52 this is t + floor(a) + c with
// c = [frac(a) >= 1 - 2^(k-53)], k = floor(log2(t + a)): the correction depends on the running
// total only through its binade.  So one pass computes, per block of SD_BLOCK records, F = sum of
// floor(a) and the cumulative histogram cum[k] = #{ i : kmin_i <= k } (kmin_i = 53+ceil(log2(1-frac)));
// a single-CTA resolver then walks the blocks with exact integer arithmetic, 8192 blocks per step,
// and only blocks that really straddle a power of two are re-read element by element.
// Totals >= 2^52 leave the closed form: the host then runs the literal sequential kernel.
// =============================================================================================
constexpr int SD_BLOCK = 8192;
constexpr int SD_THREADS = 256;
constexpr int SD_K = 52;

__device__ __forceinline__ int binade_of(double s)   // floor(log2(s)) for s >= 1, -1 below
{
  if (!(s >= 1.0)) return -1;
  return (int)((__double_as_longlong(s) >> 52) & 0x7ff) - 1023;
}

// a = (x-mean)^2 exactly as the reference computes it; returns floor(a) and kmin (255 = never)
__device__ __forceinline__ void sd_elem(int isz, double mean, double &a, long long &fa, unsigned &kmin)
{
  double x = (double)(isz < 0 ? -isz : isz);
  double d = __dsub_rn(x, mean);
  a = __dmul_rn(d, d);
  double fl = floor(a);
  fa = (long long)fl;
  double frac = a - fl;                 // exact
  kmin = 255u;
  if (frac >= 0.5) {
    double om = 1.0 - frac;             // exact for frac >= 0.5
    long long b = __double_as_longlong(om);
    int e = (int)((b >> 52) & 0x7ff) - 1023;
    int ce = e + ((b & 0xFFFFFFFFFFFFFll) != 0 ? 1 : 0);
    int km = 53 + ce;
    if (km < 0) km = 0;
    if (km < SD_K) kmin = (unsigned)km;
  }
}

// |isize| takes few distinct values, and floor(a), kmin depend on it alone once the mean is known: a 64 Ki
// entry table (kmin in the top byte, floor(a) below; 512 KB, L2/L1 resident) turns the per-record FP64
// arithmetic of the streaming pass into one lookup, which makes the pass HBM-bound again.
constexpr int SD_LUT = 65536;
__device__ __noinline__ unsigned long long sd_entry_slow(int isz, double mean)
{
  double a; long long fa; unsigned km;
  sd_elem(isz, mean, a, fa, km);
  return ((unsigned long long)km << 56) | ((unsigned long long)fa & 0x00ffffffffffffffull);
}
__global__ void sd_build_lut(double mean, unsigned long long *__restrict__ lut)
{
  int x = blockIdx.x * blockDim.x + threadIdx.x;
  if (x >= SD_LUT) return;
  double a; long long fa; unsigned km;
  sd_elem(x, mean, a, fa, km);
  lut[x] = ((unsigned long long)km << 56) | ((unsigned long long)fa & 0x00ffffffffffffffull);
}

__global__ void __launch_bounds__(SD_THREADS)
sd_block_stats(const uint8_t *__restrict__ cls, ISizeCol isz, long long n, double mean, const unsigned long long *__restrict__ lut,
               long long *__restrict__ blkF, uint32_t *__restrict__ blkCum /*[nb][SD_K]*/, uint32_t *__restrict__ blkN, double *__restrict__ blkAmax)
{
  __shared__ unsigned hist[SD_K];
  __shared__ unsigned long long sh64[33];
  __shared__ unsigned sh32[33];
  __shared__ double shd[33];
  if (threadIdx.x < SD_K) hist[threadIdx.x] = 0;
  __syncthreads();
  long long base = (long long)blockIdx.x * SD_BLOCK;
  unsigned long long F = 0, famax = 0;
  unsigned cnt = 0;
  unsigned hot = 0;        // per-thread counts of the three hot bins 51 / 50 / 49, 10 bits each (<= 32 records per thread)
  for (int g = 0; g < SD_BLOCK / (SD_THREADS * 4); ++g) {
    long long i = base + (long long)g * (SD_THREADS * 4) + threadIdx.x * 4;
    unsigned char c[4];
    int s[4];
    if (i + 3 < n) {
      uchar4 c4 = *reinterpret_cast<const uchar4 *>(cls + i);
      c[0] = c4.x; c[1] = c4.y; c[2] = c4.z; c[3] = c4.w;
      if (isz.h) { short4 h4 = *reinterpret_cast<const short4 *>(isz.h + i); s[0] = h4.x; s[1] = h4.y; s[2] = h4.z; s[3] = h4.w; }
      else { int4 s4 = *reinterpret_cast<const int4 *>(isz.w + i); s[0] = s4.x; s[1] = s4.y; s[2] = s4.z; s[3] = s4.w; }
    } else {
      for (int k = 0; k < 4; ++k) { c[k] = (i + k < n) ? cls[i + k] : 0; s[k] = (i + k < n) ? isz.at(i + k) : 0; }
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      if (c[k] & CL_INSERT) {
        unsigned x = (unsigned)(s[k] < 0 ? -s[k] : s[k]);
        unsigned long long e = (x < (unsigned)SD_LUT) ? __ldg(lut + x) : sd_entry_slow(s[k], mean);   // the slow path is a real call, not predicated code
        unsigned long long fa = e & 0x00ffffffffffffffull;
        unsigned km = (unsigned)(e >> 56);
        F += fa;
        ++cnt;
        famax = fa > famax ? fa : famax;
        hot += (km == 51u ? 1u : 0u) + (km == 50u ? (1u << 10) : 0u) + (km == 49u ? (1u << 20) : 0u);
        if (km < 49u) atomicAdd(&hist[km], 1u);
      }
    }
  }
  hot = bk::warp_sum(hot);               // <= 1024 per field per warp: no carry between the 10-bit fields
  if ((threadIdx.x & 31) == 0) {
    unsigned h51 = hot & 1023u, h50 = (hot >> 10) & 1023u, h49 = hot >> 20;
    if (h51) atomicAdd(&hist[51], h51);
    if (h50) atomicAdd(&hist[50], h50);
    if (h49) atomicAdd(&hist[49], h49);
  }
  double amax = (double)(famax + 1);          // upper bound of a: only used to bound the block's binade
  unsigned long long totF;
  bk::block_excl_scan<unsigned long long>(F, sh64, totF);
  unsigned totN;
  bk::block_excl_scan<unsigned>(cnt, sh32, totN);
  // block max of amax
  for (int o = 16; o; o >>= 1) amax = fmax(amax, __shfl_xor_sync(0xffffffffu, amax, o));
  if ((threadIdx.x & 31) == 0) shd[threadIdx.x >> 5] = amax;
  __syncthreads();
  if (threadIdx.x == 0) {
    double m = 0.0;
    for (int w = 0; w < SD_THREADS / 32; ++w) m = fmax(m, shd[w]);
    blkAmax[blockIdx.x] = m;
    blkF[blockIdx.x] = (long long)totF;
    blkN[blockIdx.x] = totN;
  }
  // cumulative histogram by two warps (a serial 52-step loop on one thread used to be the longest part of the block)
  if (threadIdx.x < 64) {
    unsigned k = threadIdx.x;
    unsigned v = k < SD_K ? hist[k] : 0u;
    unsigned inc = bk::warp_incl_scan(v);
    if (k == 31) sh32[0] = inc;
    __syncwarp();
    // the second warp adds the first warp's total after the barrier below
    if (k < 32) blkCum[(size_t)blockIdx.x * SD_K + k] = inc;
    else sh32[1 + (k - 32)] = inc;
  }
  __syncthreads();
  if (threadIdx.x >= 32 && threadIdx.x < SD_K) blkCum[(size_t)blockIdx.x * SD_K + threadIdx.x] = sh32[0] + sh32[1 + (threadIdx.x - 32)];
}

// single CTA of SDR_T threads (256 threads x 16 blocks per step measured slower than 1024 x 8).  out[0] = sd_total, out[1] = out-of-regime flag.
constexpr int SDR_T = 1024;
__global__ void __launch_bounds__(SDR_T)
sd_resolve(const uint8_t *__restrict__ cls, ISizeCol isz, long long n, double mean, int nb,
           const long long *__restrict__ blkF, const uint32_t *__restrict__ blkCum, const uint32_t *__restrict__ blkN,
           const double *__restrict__ blkAmax, long long t_in, long long *__restrict__ out)
{
  extern __shared__ unsigned char dyn[];
  double *sa = reinterpret_cast<double *>(dyn);                  // [SD_BLOCK]   a_i, -1 = ineligible
  unsigned char *skm = dyn + (size_t)SD_BLOCK * 8;               // [SD_BLOCK]   kmin_i
  __shared__ long long sh_scan[33];
  __shared__ long long sh_t;
  __shared__ int sh_j, sh_q, sh_oor, sh_k;
  if (threadIdx.x == 0) { sh_t = t_in; sh_j = 0; sh_oor = 0; }
  __syncthreads();
  constexpr int PB = 8;                     // blocks per thread and step: 8192 blocks per step
  while (true) {
    int j0 = sh_j;
    long long t0 = sh_t;
    if (j0 >= nb || sh_oor) break;
    int k0 = binade_of((double)t0);
    int jb = j0 + (int)threadIdx.x * PB;
    long long dl[PB];
    long long delta = 0;
#pragma unroll
    for (int i = 0; i < PB; ++i) {
      int j = jb + i;
      long long v = 0;
      if (j < nb) {
        v = blkF[j];
        if (k0 >= 0 && k0 < SD_K) v += blkCum[(size_t)j * SD_K + k0];
      }
      dl[i] = v; delta += v;
    }
    long long tot;
    long long tstart = t0 + bk::block_excl_scan<long long>(delta, sh_scan, tot);
    // a block is valid iff every s in it stays in binade k0
    int first_bad = SDR_T * PB;
    long long tend_of[PB];
    {
      long long ts = tstart;
#pragma unroll
      for (int i = 0; i < PB; ++i) {
        int j = jb + i;
        bool valid = true;
        if (j < nb) {
          unsigned bn = blkN[j];
          double upper = (double)(ts + dl[i] + (long long)bn + 2) + blkAmax[j] * 1.000000001 + 2.0;
          valid = (bn == 0) || (k0 < SD_K && binade_of((double)ts) == k0 && binade_of(upper) == k0);
          if (bn != 0 && k0 >= SD_K) valid = false;
          if (!valid && first_bad == SDR_T * PB) first_bad = (int)threadIdx.x * PB + i;
        }
        ts += dl[i];
        tend_of[i] = ts;
      }
    }
    if (threadIdx.x == 0) sh_q = SDR_T * PB;
    __syncthreads();
    if (first_bad < SDR_T * PB) atomicMin(&sh_q, first_bad);
    __syncthreads();
    int q = sh_q;
    int nvalid = min(q, nb - j0);          // blocks j0 .. j0+nvalid-1 are final
    __syncthreads();
    if (nvalid > 0 && (nvalid - 1) / PB == (int)threadIdx.x) {
      long long te = tend_of[0];
#pragma unroll
      for (int i = 1; i < PB; ++i) if ((nvalid - 1) % PB == i) te = tend_of[i];
      sh_t = te; sh_j = j0 + nvalid;
    }
    __syncthreads();
    if (q >= SDR_T * PB || j0 + q >= nb) continue;
    // block jq = j0+q is either the first block of a new binade or a real straddler
    int jq = j0 + q;
    long long t = sh_t;
    {
      double upper = (double)(t + blkF[jq] + (long long)blkN[jq] + 2) + blkAmax[jq] * 1.000000001 + 2.0;
      int ka = binade_of((double)t), kb = binade_of(upper);
      if (ka == kb && ka < SD_K && q > 0) continue;   // clean block of the next binade: restart the chunk there
    }
    // ---- exact element-level evaluation of block jq ----
    long long base = (long long)jq * SD_BLOCK;
    int m = (int)min((long long)SD_BLOCK, n - base);
    for (int e = threadIdx.x; e < SD_BLOCK; e += SDR_T) {
      double a = -1.0; unsigned km = 255u;
      if (e < m && (cls[base + e] & CL_INSERT)) { long long fa; sd_elem(isz.at(base + e), mean, a, fa, km); }
      sa[e] = a; skm[e] = (unsigned char)km;
    }
    __syncthreads();
    constexpr int PER = SD_BLOCK / SDR_T;
    int p = 0;
    while (p < m) {
      // first eligible element at or after p defines the current binade
      if (threadIdx.x == 0) sh_q = SD_BLOCK;
      __syncthreads();
      {
        int lo = threadIdx.x * PER, best = SD_BLOCK;
        for (int e = lo + PER - 1; e >= lo; --e) if (e >= p && e < m && sa[e] >= 0.0) best = e;
        if (best < SD_BLOCK) atomicMin(&sh_q, best);
      }
      __syncthreads();
      int pe = sh_q;
      if (pe >= SD_BLOCK) break;                       // no eligible element left
      __syncthreads();
      if (threadIdx.x == 0) { sh_k = binade_of((double)t + sa[pe]); sh_q = SD_BLOCK; }
      __syncthreads();
      int k = sh_k;
      if (k >= SD_K) { if (threadIdx.x == 0) sh_oor = 1; __syncthreads(); break; }
      // per-thread increments over its PER consecutive elements (restricted to e >= pe)
      int lo = threadIdx.x * PER;
      long long loc = 0;
      for (int e = lo; e < lo + PER; ++e)
        if (e >= pe && e < m && sa[e] >= 0.0) loc += (long long)floor(sa[e]) + ((k >= 0 && skm[e] <= k) ? 1 : 0);
      long long tt;
      long long run = t + bk::block_excl_scan<long long>(loc, sh_scan, tt);
      int cross = SD_BLOCK;
      for (int e = lo; e < lo + PER; ++e)
        if (e >= pe && e < m && sa[e] >= 0.0) {
          if (e > pe && binade_of((double)run + sa[e]) > k && cross == SD_BLOCK) cross = e;
          run += (long long)floor(sa[e]) + ((k >= 0 && skm[e] <= k) ? 1 : 0);
        }
      if (cross < SD_BLOCK) atomicMin(&sh_q, cross);
      __syncthreads();
      int qx = sh_q;
      // add the increments of [pe, qx)
      long long part = 0;
      for (int e = lo; e < lo + PER; ++e)
        if (e >= pe && e < qx && e < m && sa[e] >= 0.0) part += (long long)floor(sa[e]) + ((k >= 0 && skm[e] <= k) ? 1 : 0);
      long long ptot;
      bk::block_excl_scan<long long>(part, sh_scan, ptot);
      t += ptot;
      p = qx;
      __syncthreads();
    }
    if (threadIdx.x == 0) { sh_t = t; sh_j = jq + 1; }
    __syncthreads();
  }
  if (threadIdx.x == 0) { out[0] = sh_t; out[1] = sh_oor; }
}

// literal sequential replay (one thread); only used when the total leaves the closed-form regime
__global__ void sd_sequential(const uint8_t *__restrict__ cls, ISizeCol isz, long long n, double mean, long long t_in, long long *out)
{
  if (blockIdx.x || threadIdx.x) return;
  long long t = t_in;
  for (long long i = 0; i < n; ++i)
    if (cls[i] & CL_INSERT) {
      int s = isz.at(i);
      double x = (double)(s < 0 ? -s : s);
      double d = __dsub_rn(x, mean);
      t = (long long)__dadd_rn((double)t, __dmul_rn(d, d));
    }
  out[0] = t; out[1] = 0;
}

// ---- the common case in ONE streaming pass -----------------------------------------------------------------
// With S, N and the sum of squares from K1 the final total is bounded before the pass: T <= T_ub, so every running
// total lies in a binade k <= K = floor(log2(T_ub)).  An element then needs a correction only if
// frac(a) >= 1 - 2^(K-53) =: thr.  sd_fast adds up floor(a) and COUNTS such elements (E).  E = 0 (no insert size
// whose squared deviation has a fraction that close to 1 -- |isize| takes a few hundred values, K is ~39 for a 30x
// genome, so this is the normal case) means total = sum floor(a) exactly, independent of the order: no block tables,
// no resolver, and in the multi-GPU path no rank-to-rank chain.  E > 0 falls back to the general path above.
// Arithmetic per record: 6 FP64 instructions, no conversions -- x -> double by the 2^52 bit pattern, floor(a) by a
// round-down add of 2^52 (exact for 0 <= a < 2^51; larger values raise the out-of-regime flag).
// out[0] += sum floor(a), out[1] += E, out[2] |= out of regime.
// floor(a) and the correction test of one |isize| (FP64 path): returns floor(a), sets rare / oor
__device__ __forceinline__ unsigned long long sd_fast_eval(unsigned x, double mean, double thr, bool &rare, bool &oor)
{
  const double M52 = 4503599627370496.0;
  double xd = __dsub_rn(__hiloint2double(0x43300000, (int)x), M52);      // exact for x < 2^32
  double d = __dsub_rn(xd, mean);
  double a = __dmul_rn(d, d);
  double sft = __dadd_rd(a, M52);                                         // 2^52 + floor(a)
  double fr = __dsub_rn(a, __dsub_rn(sft, M52));                          // frac(a), exact
  rare = fr >= thr;
  oor = !(a < 2251799813685248.0);
  return (unsigned long long)__double_as_longlong(sft) & 0xFFFFFFFFFFFFFull;
}
// |isize| takes few values, all near the mean: every CTA first tabulates floor(a) for the SDF_WIN values around the mean in
// shared memory (32-bit entries -- random lanes hit 32 banks; 0xffffffff = does not fit / needs the full evaluation), so
// the streaming loop costs one shared load and a handful of integer instructions per record instead of six FP64 ones
// (the all-FP64 version ran at 0.47 of the HBM peak: FP64-pipe bound).
constexpr int SDF_WIN = 4096;
template <bool NARROW>
__global__ void __launch_bounds__(256)
sd_fast(const uint8_t *__restrict__ cls, const int32_t *__restrict__ isize, const int16_t *__restrict__ isize16, long long n, double mean, double thr,
        unsigned long long *__restrict__ out)
{
  // tab[0 .. WIN) = floor(a) of |isize| = xlo + k; tab[WIN] = "outside the window / needs the full evaluation" (also used for
  // entries that do not fit: rare, out of regime, or >= 2^28 so that eight entries add up in 32 bits); tab[WIN + 1] = 0 is
  // where records that do not pass the insert predicate are sent -- no branch per record
  __shared__ uint32_t tab[SDF_WIN + 2];
  const double mc = mean < 0.0 ? 0.0 : (mean > 2.0e9 ? 2.0e9 : mean);      // NaN -> 0 as well
  const unsigned xlo = (unsigned)mc > (unsigned)(SDF_WIN / 2) ? (unsigned)mc - (unsigned)(SDF_WIN / 2) : 0u;
  for (int k = threadIdx.x; k < SDF_WIN; k += blockDim.x) {
    bool rare, oor;
    unsigned long long fa = sd_fast_eval(xlo + (unsigned)k, mean, thr, rare, oor);
    tab[k] = (rare || oor || fa >= (1ull << 28)) ? 0xffffffffu : (uint32_t)fa;
  }
  if (threadIdx.x == 0) { tab[SDF_WIN] = 0xffffffffu; tab[SDF_WIN + 1] = 0u; }
  __syncthreads();
  unsigned long long F = 0; unsigned E = 0, oorf = 0;
  const long long ngroups = (n + 7) / 8;
  for (long long gi = (long long)blockIdx.x * blockDim.x + threadIdx.x; gi < ngroups; gi += (long long)gridDim.x * blockDim.x) {
    long long i = gi * 8;
    unsigned cm;                                         // bit 8k = record k passes the insert predicate
    int sv[8];
    if (i + 7 < n) {
      uint2 c8 = *reinterpret_cast<const uint2 *>(cls + i);
      cm = (c8.x & 0x01010101u) | ((c8.y & 0x01010101u) << 1);     // records 0-3 at bits 0,8,16,24; records 4-7 at bits 1,9,17,25
      if (NARROW) {
        uint4 h8 = *reinterpret_cast<const uint4 *>(isize16 + i);
        sv[0] = (int)(short)(h8.x & 0xffffu); sv[1] = (int)h8.x >> 16; sv[2] = (int)(short)(h8.y & 0xffffu); sv[3] = (int)h8.y >> 16;
        sv[4] = (int)(short)(h8.z & 0xffffu); sv[5] = (int)h8.z >> 16; sv[6] = (int)(short)(h8.w & 0xffffu); sv[7] = (int)h8.w >> 16;
      } else {
        int4 a4 = *reinterpret_cast<const int4 *>(isize + i), b4 = *reinterpret_cast<const int4 *>(isize + i + 4);
        sv[0] = a4.x; sv[1] = a4.y; sv[2] = a4.z; sv[3] = a4.w; sv[4] = b4.x; sv[5] = b4.y; sv[6] = b4.z; sv[7] = b4.w;
      }
    } else {
      cm = 0;
      for (int k = 0; k < 8; ++k) {
        bool on = i + k < n && (cls[i + k] & CL_INSERT);
        sv[k] = (i + k < n) ? (NARROW ? (int)isize16[i + k] : isize[i + k]) : 0;
        if (on) cm |= k < 4 ? (1u << (8 * k)) : (2u << (8 * (k - 4)));
      }
    }
    unsigned part = 0;                                   // eight table entries < 2^28 each
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const unsigned bit = k < 4 ? (1u << (8 * k)) : (2u << (8 * (k - 4)));
      unsigned x = (unsigned)(sv[k] < 0 ? -sv[k] : sv[k]);
      unsigned w = min(x - xlo, (unsigned)SDF_WIN);     // x < xlo wraps to a huge value: the window-miss entry
      uint32_t t = tab[(cm & bit) ? w : (unsigned)(SDF_WIN + 1)];
      if (t != 0xffffffffu) part += t;
      else {
        bool rare, oor;
        F += sd_fast_eval(x, mean, thr, rare, oor);
        E += rare ? 1u : 0u; oorf |= oor ? 1u : 0u;
      }
    }
    F += part;
  }
  F = bk::warp_sum(F); E = bk::warp_sum(E); oorf = bk::warp_sum(oorf);
  if ((threadIdx.x & 31) == 0) {
    if (F) atomicAdd(out, F);
    if (E) atomicAdd(out + 1, (unsigned long long)E);
    if (oorf) atomicOr(out + 2, 1ull);
  }
}

// =============================================================================================
// K2: mate join.  Candidates (ordered by file position) are sorted by the low 64 bits of the name
// hash with a stable radix sort, so the records sharing a name sit in one run in file order.  The
// reference's std::map protocol (store first, pair-and-erase on the second, src/BreakID.cc:1424-1494)
// pairs run positions (0,1), (2,3), ...: the odd one is the "current" record, the even one the
// stored mate.
// =============================================================================================
// candidate records are gathered once into a compact array (bkid_cand, 48 B): the sort, the run
// detection and the pair emission then touch two coalesced 48-byte rows per pair instead of eleven
// scattered column reads, and the same array is what ranks exchange in the multi-GPU path.
// slot of record i in the sparse table (x_rec ascending), or -1
__device__ __forceinline__ long long x_slot_of(const uint32_t *__restrict__ x_rec, long long n_x, uint32_t i)
{
  long long lo = 0, hi = n_x;
  while (lo < hi) { long long m = (lo + hi) >> 1; if (x_rec[m] < i) lo = m + 1; else hi = m; }
  return (lo < n_x && x_rec[lo] == i) ? lo : -1;
}

// ---- candidates straight from the sparse mate/name table -------------------------------------------------------
// Every candidate (:1419-1420) is by construction listed in the sparse table (it is not a proper pair), and the table is
// in file order: one pass over its ~1 % entries yields the compact candidate array in file order -- no sweep over the
// class bytes of all records, no search.  kx_count: candidates per 1024-entry tile (and the table's sanity: strictly
// ascending record indices inside the batch); kx_write: ordered compaction into bkid_cand rows + the join's sort keys.
constexpr int KX_THREADS = 256;
constexpr int KX_ITEMS = 2;
constexpr int KX_TILE = KX_THREADS * KX_ITEMS;

__global__ void __launch_bounds__(KX_THREADS) kx_count(const uint32_t *__restrict__ x_rec, long long n_x, const uint8_t *__restrict__ cand_bits, long long n,
                                                       uint32_t *__restrict__ tile_cnt, uint8_t *__restrict__ is_cand /* [n_x / KX_ITEMS]: KX_ITEMS flag bits per thread */, int *__restrict__ bad)
{
  __shared__ unsigned sh32[33];
  long long j0 = (long long)blockIdx.x * KX_TILE + threadIdx.x * KX_ITEMS;
  unsigned cnt = 0, bits = 0;
  uint32_t r[KX_ITEMS]; unsigned char c[KX_ITEMS];
  uint32_t rprev = j0 > 0 && j0 < n_x ? x_rec[j0 - 1] : 0u;
#pragma unroll
  for (int k = 0; k < KX_ITEMS; ++k) r[k] = j0 + k < n_x ? x_rec[j0 + k] : 0xffffffffu;
#pragma unroll
  for (int k = 0; k < KX_ITEMS; ++k)      // independent loads, issued together; neighbouring entries share bitmap sectors (1 bit per record)
    c[k] = (j0 + k < n_x && (long long)r[k] < n) ? (unsigned char)(((cand_bits[r[k] >> 3] >> (r[k] & 7u)) & 1u) ? CL_CAND : 0) : 0;
#pragma unroll
  for (int k = 0; k < KX_ITEMS; ++k) {
    long long j = j0 + k;
    if (j < n_x) {
      if ((long long)r[k] >= n || (j > 0 && rprev >= r[k])) atomicExch(bad, 1);
      else if (c[k] & CL_CAND) { ++cnt; bits |= 1u << k; }
      rprev = r[k];
    }
  }
  if (j0 < n_x) is_cand[j0 / KX_ITEMS] = (uint8_t)bits;
  unsigned tot;
  bk::block_excl_scan<unsigned>(cnt, sh32, tot);
  if (threadIdx.x == 0) tile_cnt[blockIdx.x] = tot;
}

__global__ void __launch_bounds__(KX_THREADS) kx_write(const uint32_t *__restrict__ x_rec, long long n_x, const uint8_t *__restrict__ is_cand, long long n, const uint32_t *__restrict__ tile_off,
                                                       const uint16_t *__restrict__ flag, const uint8_t *__restrict__ mapq, const int32_t *__restrict__ tid, const int32_t *__restrict__ pos,
                                                       const int32_t *__restrict__ x_mtid, const int32_t *__restrict__ x_mpos, const uint64_t *__restrict__ x_nh,
                                                       unsigned long long index_offset, bkid_cand *__restrict__ out, uint64_t *__restrict__ keys, uint32_t *__restrict__ vals)
{
  __shared__ unsigned sh32[33];
  long long j0 = (long long)blockIdx.x * KX_TILE + threadIdx.x * KX_ITEMS;
  __shared__ __align__(16) bkid_cand srow[KX_TILE];             // the tile's rows are assembled here and leave as one contiguous, coalesced range
  const unsigned bits = j0 < n_x ? (unsigned)is_cand[j0 / KX_ITEMS] : 0u;       // kx_count's verdict: the class bytes are not read again
  unsigned tot;
  unsigned loc = bk::block_excl_scan<unsigned>(__popc(bits), sh32, tot);
  const unsigned tile0 = tile_off[blockIdx.x];
  // gather the four dense fields of this thread's candidates first (independent loads), then assemble the rows
  uint32_t i4[KX_ITEMS]; int32_t t4[KX_ITEMS], p4[KX_ITEMS]; uint16_t f4[KX_ITEMS]; uint8_t m4[KX_ITEMS];
#pragma unroll
  for (int k = 0; k < KX_ITEMS; ++k) i4[k] = (bits >> k) & 1u ? x_rec[j0 + k] : 0u;
#pragma unroll
  for (int k = 0; k < KX_ITEMS; ++k)
    if ((bits >> k) & 1u) { t4[k] = tid[i4[k]]; p4[k] = pos[i4[k]]; f4[k] = flag[i4[k]]; m4[k] = mapq[i4[k]]; }
#pragma unroll
  for (int k = 0; k < KX_ITEMS; ++k)
    if ((bits >> k) & 1u) {
      long long j = j0 + k;
      bkid_cand c;
      c.name_lo = x_nh[2 * (size_t)j]; c.name_hi = x_nh[2 * (size_t)j + 1];
      c.tid = t4[k]; c.pos = p4[k]; c.mtid = x_mtid[j]; c.mpos = x_mpos[j];
      c.gidx = index_offset + i4[k];
      c.flag = f4[k]; c.mapq = m4[k];
      c._pad[0] = c._pad[1] = c._pad[2] = c._pad[3] = c._pad[4] = 0;
      srow[loc++] = c;
    }
  __syncthreads();
  const uint4 *sv = reinterpret_cast<const uint4 *>(srow);
  uint4 *ov = reinterpret_cast<uint4 *>(out + tile0);
  for (unsigned i = threadIdx.x; i < tot * 3u; i += KX_THREADS) ov[i] = sv[i];
  if (keys)
    for (unsigned i = threadIdx.x; i < tot; i += KX_THREADS) { keys[tile0 + i] = srow[i].name_lo; vals[tile0 + i] = tile0 + i; }
}

__global__ void k2_cand_keys(const bkid_cand *__restrict__ cand, long long nc, uint64_t *__restrict__ keys, uint32_t *__restrict__ vals)
{
  long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (p < nc) { keys[p] = cand[p].name_lo; vals[p] = (uint32_t)p; }
}

__device__ __forceinline__ uint32_t genome_pos(const uint32_t *__restrict__ cum, int nt, int tid, int pos)
{
  // src/util_bam.cc:57-68: sum of target_len[0..tid) (uint32 wrap) + pos; tid < 0 adds nothing
  uint32_t p = (tid > 0) ? cum[tid < nt ? tid : nt] : 0u;
  return p + (uint32_t)pos;
}

// sort key of a pair: bucket rank (high 24 bits) | global index of the second-seen mate (40 bits)
constexpr int PAIR_IDX_BITS = 40;
constexpr uint32_t NO_MATE = 0xffffffffu;

// one discordant pair from its two records: I = current (second seen), J = the stored mate (src/BreakID.cc:1428-1480)
__device__ __forceinline__ bool pair_is_discordant(const bkid_cand &I, const bkid_cand &J, double w)
{
  int ti = I.tid < 0 ? -1 : I.tid, tj = J.tid < 0 ? -1 : J.tid;
  long long pi = (long long)I.pos + 1, pj = (long long)J.pos + 1;
  long long dp = pi - pj; if (dp < 0) dp = -dp;
  return (ti != tj) || ((double)dp >= w);                     // :1428
}
__device__ __forceinline__ bkid_pair make_pair(const bkid_cand &I, const bkid_cand &J, const uint32_t *__restrict__ cum, int nt, const int32_t *__restrict__ bucket_rank)
{
  uint32_t c1 = genome_pos(cum, nt, I.tid, I.pos);            // :1431 current record's own fields
  uint32_t c2 = genome_pos(cum, nt, I.mtid, I.mpos);          // :1432 and its mate FIELDS
  bkid_pair P;
  P.name_lo = I.name_lo; P.name_hi = I.name_hi;
  int ti = I.tid < 0 ? -1 : I.tid, tj = J.tid < 0 ? -1 : J.tid;
  uint32_t pi = (uint32_t)((long long)I.pos + 1), pj = (uint32_t)((long long)J.pos + 1);
  if (c1 <= c2) {
    P.p1_flag = I.flag; P.p1_tid = ti; P.p1_pos = pi; P.p1_mapq = I.mapq;
    P.p2_flag = J.flag; P.p2_tid = tj; P.p2_pos = pj; P.p2_mapq = J.mapq;
    P.p1_chr_pos = c1; P.p2_chr_pos = c2;
  } else {
    P.p2_flag = I.flag; P.p2_tid = ti; P.p2_pos = pi; P.p2_mapq = I.mapq;
    P.p1_flag = J.flag; P.p1_tid = tj; P.p1_pos = pj; P.p1_mapq = J.mapq;
    P.p1_chr_pos = c2; P.p2_chr_pos = c1;
  }
  P.p1_strand = (P.p1_flag & F_REVERSE) ? '-' : '+';
  P.p2_strand = (P.p2_flag & F_REVERSE) ? '-' : '+';
  int a = P.p1_tid + 1, b = P.p2_tid + 1;
  P.bucket = bucket_rank[a * (nt + 1) + b];                   // rank of "chrA_chrB" among all possible names
  P.cluster = -1;
  P.orig = (uint32_t)(I.gidx & 0xffffffffull);                // order of the second-seen mate (40 bits: orig | _pad << 32)
  P._pad = (uint32_t)((I.gidx >> 32) & 0xffull);
  return P;
}

// The join proper.  (keys, vals) = (name_lo, candidate index) stably sorted on the low `group_bits` bits of name_lo, so
// all records of a read name sit in one GROUP in file order -- possibly interleaved with the few other names that share
// those bits (3.4e6 names on 32 bits: ~1e3 groups).  The thread at the head of a group walks it: a group that is not
// one name is first sorted, stably, on the full 128-bit name (insertion sort, <= cap members; this is also what
// resolves two names that share all 64 bits of name_lo); then the records of every name are taken in file order and
// paired (0,1), (2,3), ... -- the reference's std::map store / pair-and-erase protocol (src/BreakID.cc:1424-1494) --
// and mate[second seen] = stored mate for the pairs that pass the discordance test.  A larger mixed group raises
// *too_big: the caller then sorts on all 64 bits and runs the walk again.
__global__ void __launch_bounds__(256) k2_join(uint64_t *__restrict__ keys, uint32_t *__restrict__ vals, const uint32_t *__restrict__ nc_dev, uint32_t nc_host,
                                               const bkid_cand *__restrict__ cand, int group_bits, uint32_t cap, double w, uint32_t *__restrict__ mate, int *__restrict__ too_big)
{
  const uint32_t nc = nc_dev ? *nc_dev : nc_host;
  uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= nc) return;
  const uint64_t gmask = group_bits >= 64 ? ~0ull : ((1ull << group_bits) - 1ull);
  const uint64_t k0 = keys[p], gk = k0 & gmask;
  if (p > 0 && (keys[p - 1] & gmask) == gk) return;             // not the head of its group
  uint32_t e = p + 1;
  while (e < nc && (keys[e] & gmask) == gk) ++e;
  if (e - p < 2) return;                                        // a lone record has no mate
  uint64_t hi_prev = cand[vals[p]].name_hi;
  bool mixed = false;
  for (uint32_t q = p + 1; q < e && !mixed; ++q) mixed = keys[q] != k0 || cand[vals[q]].name_hi != hi_prev;
  if (mixed) {
    if (e - p > cap) { atomicExch(too_big, 1); return; }
    for (uint32_t i = p + 1; i < e; ++i) {                      // stable insertion sort on (name_lo, name_hi)
      uint64_t kl = keys[i]; uint32_t v = vals[i]; uint64_t kh = cand[v].name_hi;
      uint32_t j = i;
      while (j > p) {
        uint64_t pl = keys[j - 1], ph = cand[vals[j - 1]].name_hi;
        if (pl < kl || (pl == kl && ph <= kh)) break;
        keys[j] = pl; vals[j] = vals[j - 1]; --j;
      }
      keys[j] = kl; vals[j] = v;
    }
    hi_prev = cand[vals[p]].name_hi;
  }
  uint32_t run_start = p;
  uint64_t lo_prev = keys[p];
  for (uint32_t q = p + 1; q < e; ++q) {
    uint32_t vq = vals[q];
    uint64_t lo = keys[q], hi = cand[vq].name_hi;
    if (lo != lo_prev || hi != hi_prev) { run_start = q; lo_prev = lo; hi_prev = hi; continue; }
    if ((q - run_start) & 1u) {
      uint32_t vj = vals[q - 1];
      bkid_cand I = cand[vq], J = cand[vj];
      if (pair_is_discordant(I, J, w)) mate[vq] = vj;
    }
  }
}

__global__ void k2_mate_flags(const uint32_t *__restrict__ mate, long long nc, uint32_t *__restrict__ flag)
{
  long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (q < nc) flag[q] = mate[q] != NO_MATE ? 1u : 0u;
}

// pairs in the order of their second-seen mate (= the order in which the reference's scan emits them)
__global__ void k2_build_pairs(const uint32_t *__restrict__ mate, const uint32_t *__restrict__ off, long long nc, const bkid_cand *__restrict__ cand,
                               const uint32_t *__restrict__ cum, int nt, const int32_t *__restrict__ bucket_rank, bkid_pair *__restrict__ pairs)
{
  long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= nc) return;
  uint32_t m = mate[q];
  if (m == NO_MATE) return;
  bkid_cand I = cand[q], J = cand[m];
  pairs[off[q]] = make_pair(I, J, cum, nt, bucket_rank);
}

// ordered: the pairs already arrive in emission order (single GPU) -> key = bucket rank alone (a stable sort keeps the
// order inside a bucket); otherwise (pairs gathered from several ranks) key = bucket rank | index of the second-seen mate
__global__ void k2_pair_keys(const bkid_pair *__restrict__ pairs, long long np, int ordered, unsigned long long *__restrict__ keys, uint32_t *__restrict__ slots)
{
  long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= np) return;
  const bkid_pair &P = pairs[p];
  keys[p] = ordered ? ((unsigned long long)(unsigned)P.bucket << PAIR_IDX_BITS)
                    : (((unsigned long long)(unsigned)P.bucket << PAIR_IDX_BITS) | ((unsigned long long)P._pad << 32) | (unsigned long long)P.orig);
  slots[p] = (uint32_t)p;
}

__global__ void k2_gather_pairs(const bkid_pair *__restrict__ src, const uint32_t *__restrict__ slots, const unsigned long long *__restrict__ keys,
                                long long np, bkid_pair *__restrict__ dst, uint32_t *__restrict__ bucket_head)
{
  long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= np) return;
  bkid_pair P = src[slots[p]];
  P.orig = (uint32_t)p;
  P._pad = 0;
  dst[p] = P;
  bucket_head[p] = (p == 0 || (keys[p] >> PAIR_IDX_BITS) != (keys[p - 1] >> PAIR_IDX_BITS)) ? 1u : 0u;
}

// dense bucket ids + bucket offsets
__global__ void k2_bucket_ids(bkid_pair *__restrict__ pairs, const uint32_t *__restrict__ head, const uint32_t *__restrict__ head_excl, long long np,
                              uint32_t *__restrict__ bucket_off, int32_t *__restrict__ bucket_rank_of)
{
  long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= np) return;
  uint32_t b = head_excl[p] - (head[p] ? 0u : 1u);
  if (head[p]) { bucket_off[b] = (uint32_t)p; bucket_rank_of[b] = pairs[p].bucket; }
  pairs[p].bucket = (int32_t)b;
}

// =============================================================================================
// K3: replay of libstdc++ std::sort (introsort) on (key, value) segments -- see the model and its
// proof obligations in oracle/oracle.cc (orc_model_sort_perm).  Level-synchronous: one CTA per
// active segment does median-of-3 + the data-parallel form of __unguarded_partition; segments of
// <= 16 elements are finished by one thread each (stable insertion sort); depth-exhausted segments
// run the literal heapsort on one thread.
// =============================================================================================
struct Seg { uint32_t f, l; int depth; };
constexpr int IS_THREADS = 512;
constexpr int IS_ITEMS = 4;
constexpr uint32_t IS_SMALL = 1024;     // segments up to this size are finished by one warp in shared memory

__device__ void seg_insertion_sort(uint32_t *key, uint32_t *val, uint32_t f, uint32_t l)
{
  for (uint32_t i = f + 1; i < l; ++i) {
    uint32_t k = key[i], v = val[i];
    uint32_t j = i;
    while (j > f && k < key[j - 1]) { key[j] = key[j - 1]; val[j] = val[j - 1]; --j; }
    key[j] = k; val[j] = v;
  }
}

__device__ void seg_heapsort(uint32_t *key, uint32_t *val, uint32_t f, uint32_t l)
{
  // std::__partial_sort(first,last,last): __make_heap + __sort_heap (libstdc++ bits/stl_heap.h)
  long n = (long)l - (long)f;
  uint32_t *K = key + f, *V = val + f;
  auto adjust = [&](long hole, long len, uint32_t vk, uint32_t vv) {
    const long top = hole;
    long child = hole;
    while (child < (len - 1) / 2) {
      child = 2 * (child + 1);
      if (K[child] < K[child - 1]) child--;
      K[hole] = K[child]; V[hole] = V[child];
      hole = child;
    }
    if ((len & 1) == 0 && child == (len - 2) / 2) {
      child = 2 * (child + 1);
      K[hole] = K[child - 1]; V[hole] = V[child - 1];
      hole = child - 1;
    }
    long parent = (hole - 1) / 2;
    while (hole > top && K[parent] < vk) {
      K[hole] = K[parent]; V[hole] = V[parent];
      hole = parent;
      parent = (hole - 1) / 2;
    }
    K[hole] = vk; V[hole] = vv;
  };
  if (n < 2) return;
  for (long parent = (n - 2) / 2;; --parent) {
    adjust(parent, n, K[parent], V[parent]);
    if (parent == 0) break;
  }
  for (long last = n - 1; last > 0; --last) {
    uint32_t vk = K[last], vv = V[last];
    K[last] = K[0]; V[last] = V[0];
    adjust(0, last, vk, vv);
  }
}

// A segment above IS_BIG elements is partitioned by several CTAs (is_big_part / is_big_swap below): one CTA streams a
// 200 K element bucket at ~0.4 ms per level, and the skewed partitions the replay must reproduce keep such a segment
// alive for 20+ levels (measured: 16 ms of is_level on one rank of the 8-GPU workload).
struct BigSeg { uint32_t f, l; int depth; uint32_t tile_base, ntiles, pv, ready, nL, nR, _pad; };
constexpr uint32_t IS_BIG = 49152;       // above the largest chr-pair bucket of a 30x genome (~35 K pairs): the single-GPU step never pays for the extra launches
constexpr uint32_t IS_BTILE = 2048;     // elements per tile of a big segment (= IS_THREADS * IS_ITEMS)
__device__ __forceinline__ void big_route(const Seg &s, BigSeg *big, unsigned long long *n_big /* count << 32 | tiles */)
{
  uint32_t nt = (s.l - s.f - 1 + IS_BTILE - 1) / IS_BTILE;
  unsigned long long old = atomicAdd(n_big, (1ull << 32) | (unsigned long long)nt);      // list slot and tile range in ONE atomic: slots are ordered by tile_base
  big[old >> 32] = BigSeg{s.f, s.l, s.depth, (uint32_t)old, nt, 0u, 0u, 0u, 0u, 0u};
}
__device__ __forceinline__ void seg_route(const Seg &s, Seg *act, unsigned *n_act, Seg *small, unsigned *n_small, Seg *term, unsigned *n_term,
                                          BigSeg *big = nullptr, unsigned long long *n_big = nullptr)
{
  uint32_t sz = s.l - s.f;
  if (big && sz > IS_BIG) big_route(s, big, n_big);
  else if (sz > IS_SMALL) act[atomicAdd(n_act, 1u)] = s;
  else if (sz > 16) small[atomicAdd(n_small, 1u)] = s;
  else if (sz >= 2) term[atomicAdd(n_term, 1u)] = s;
}

// roots: one segment per bucket
__global__ void is_init_roots(const uint32_t *__restrict__ seg_off, int nseg, Seg *__restrict__ act, unsigned *__restrict__ n_act,
                              Seg *__restrict__ small, unsigned *__restrict__ n_small, Seg *__restrict__ term, unsigned *__restrict__ n_term,
                              BigSeg *__restrict__ big, unsigned long long *__restrict__ n_big)
{
  int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= nseg) return;
  uint32_t f = seg_off[s], l = seg_off[s + 1];
  uint32_t n = l - f;
  if (n < 2) return;
  int lg = 31 - __clz(n);
  seg_route(Seg{f, l, 2 * lg}, act, n_act, small, n_small, term, n_term, big, n_big);
}

// one warp per small segment, everything in shared memory: the same partition scheme as is_level
// (L / R lists via ballots), an explicit stack instead of levels, terminal (<= 16) segments finished
// by one lane each (stable insertion sort), depth-exhausted segments by the literal heapsort.
constexpr int ISS_WARPS = 2;
__global__ void __launch_bounds__(ISS_WARPS * 32) is_small(uint32_t *__restrict__ key, uint32_t *__restrict__ val, const Seg *__restrict__ small, const unsigned *__restrict__ n_small_p)
{
  __shared__ uint32_t sk[ISS_WARPS][IS_SMALL], sv[ISS_WARPS][IS_SMALL];
  __shared__ uint16_t sL[ISS_WARPS][IS_SMALL], sR[ISS_WARPS][IS_SMALL];
  __shared__ uint16_t tf[ISS_WARPS][IS_SMALL / 2], tl[ISS_WARPS][IS_SMALL / 2];
  __shared__ int stf[ISS_WARPS][64], stl[ISS_WARPS][64], stdp[ISS_WARPS][64];
  const unsigned w = threadIdx.x >> 5, lane = threadIdx.x & 31, ltmask = (1u << lane) - 1u;
  uint32_t *K = sk[w], *V = sv[w];
  uint16_t *L = sL[w], *R = sR[w];
  unsigned n_small = *n_small_p;
  for (unsigned si = blockIdx.x * ISS_WARPS + w; si < n_small; si += gridDim.x * ISS_WARPS) {
    Seg s = small[si];
    int n = (int)(s.l - s.f);
    for (int i = lane; i < n; i += 32) { K[i] = key[s.f + i]; V[i] = val[s.f + i]; }
    int sp = 1, nt = 0;
    if (lane == 0) { stf[w][0] = 0; stl[w][0] = n; stdp[w][0] = s.depth; }
    __syncwarp();
    while (sp) {
      --sp;
      int first = stf[w][sp], last = stl[w][sp], d = stdp[w][sp];
      __syncwarp();
      while (last - first > 16) {
        if (d == 0) { if (lane == 0) seg_heapsort(K, V, (uint32_t)first, (uint32_t)last); __syncwarp(); first = last; break; }
        --d;
        if (lane == 0) {
          int mid = first + (last - first) / 2, A = first + 1, B = mid, C = last - 1, med;
          uint32_t ka = K[A], kb = K[B], kc = K[C];
          if (ka < kb) { if (kb < kc) med = B; else if (ka < kc) med = C; else med = A; }
          else if (ka < kc) med = A;
          else if (kb < kc) med = C;
          else med = B;
          uint32_t tk = K[first], tv = V[first];
          K[first] = K[med]; V[first] = V[med]; K[med] = tk; V[med] = tv;
        }
        __syncwarp();
        uint32_t pv = K[first];
        int lo = first + 1, cnt = last - lo, nL = 0, nR = 0;
        for (int b = 0; b < cnt; b += 32) {
          int e = b + (int)lane;
          bool isL = e < cnt && !(K[lo + e] < pv);
          unsigned m = __ballot_sync(0xffffffffu, isL);
          if (isL) L[nL + __popc(m & ltmask)] = (uint16_t)(lo + e);
          nL += __popc(m);
          bool isR = e < cnt && !(pv < K[last - 1 - e]);
          m = __ballot_sync(0xffffffffu, isR);
          if (isR) R[nR + __popc(m & ltmask)] = (uint16_t)(last - 1 - e);
          nR += __popc(m);
        }
        __syncwarp();
        int mn = nL < nR ? nL : nR, Kc = 0;
        for (int b = 0; b < mn; b += 32) {
          int k = b + (int)lane;
          unsigned m = __ballot_sync(0xffffffffu, k < mn && L[k] < R[k]);
          Kc += __popc(m);
          if (m != 0xffffffffu) break;
        }
        for (int k = lane; k < Kc; k += 32) {
          int a = L[k], b2 = R[k];
          uint32_t tk = K[a], tv = V[a];
          K[a] = K[b2]; V[a] = V[b2]; K[b2] = tk; V[b2] = tv;
        }
        int rprev = Kc ? (int)R[Kc - 1] : last;
        int cut = (Kc < nL && (int)L[Kc] < rprev) ? (int)L[Kc] : rprev;
        __syncwarp();
        // right part goes on the stack (or to the terminal list), continue with the left part
        int rs = last - cut;
        if (rs > 16) { if (lane == 0) { stf[w][sp] = cut; stl[w][sp] = last; stdp[w][sp] = d; } ++sp; }
        else if (rs >= 2) { if (lane == 0) { tf[w][nt] = (uint16_t)cut; tl[w][nt] = (uint16_t)last; } ++nt; }
        last = cut;
        __syncwarp();
      }
      if (last - first >= 2) { if (lane == 0) { tf[w][nt] = (uint16_t)first; tl[w][nt] = (uint16_t)last; } ++nt; }
      __syncwarp();
    }
    for (int t = lane; t < nt; t += 32) seg_insertion_sort(K, V, tf[w][t], tl[w][t]);
    __syncwarp();
    for (int i = lane; i < n; i += 32) { key[s.f + i] = K[i]; val[s.f + i] = V[i]; }
    __syncwarp();
  }
}

__global__ void __launch_bounds__(IS_THREADS)
is_level(uint32_t *__restrict__ key, uint32_t *__restrict__ val, const Seg *__restrict__ act, const unsigned *__restrict__ n_act_p,
         Seg *__restrict__ nxt, unsigned *__restrict__ n_nxt, Seg *__restrict__ small, unsigned *__restrict__ n_small,
         Seg *__restrict__ term, unsigned *__restrict__ n_term, uint32_t *__restrict__ scrL, uint32_t *__restrict__ scrR,
         Seg *__restrict__ heap, unsigned *__restrict__ n_heap)
{
  __shared__ unsigned sh32[33];
  __shared__ uint32_t sh_p;
  __shared__ unsigned sh_K;
  unsigned n_act = *n_act_p;
  for (unsigned si = blockIdx.x; si < n_act; si += gridDim.x) {
    Seg s = act[si];
    uint32_t f = s.f, l = s.l;
    if (s.depth == 0) {                                        // depth budget spent: the literal heapsort, done by is_heap at the end of the sort
      if (threadIdx.x == 0) heap[atomicAdd(n_heap, 1u)] = s;
      continue;
    }
    if (threadIdx.x == 0) {
      // __move_median_to_first(first, first+1, mid, last-1)
      uint32_t mid = f + (l - f) / 2, A = f + 1, B = mid, C = l - 1;
      uint32_t ka = key[A], kb = key[B], kc = key[C], med;
      if (ka < kb) { if (kb < kc) med = B; else if (ka < kc) med = C; else med = A; }
      else if (ka < kc) med = A;
      else if (kb < kc) med = C;
      else med = B;
      uint32_t tk = key[f], tv = val[f];
      key[f] = key[med]; val[f] = val[med];
      key[med] = tk; val[med] = tv;
      sh_p = key[f];
    }
    __syncthreads();
    uint32_t pv = sh_p;
    uint32_t lo = f + 1, cnt = l - lo;
    // L list: ascending positions with key >= pivot; R list: descending positions with key <= pivot.
    // Each thread owns IS_ITEMS consecutive elements of a tile (from the left for L, from the right for R), so
    // one pair of block scans covers IS_THREADS * IS_ITEMS elements.
    unsigned nL = 0, nR = 0;
    for (uint32_t b = 0; b < cnt; b += IS_THREADS * IS_ITEMS) {
      uint32_t e0 = b + threadIdx.x * IS_ITEMS;
      unsigned mL = 0, mR = 0, cL = 0, cR = 0;
#pragma unroll
      for (int k = 0; k < IS_ITEMS; ++k) {
        uint32_t e = e0 + k;
        if (e < cnt) {
          if (!(key[lo + e] < pv)) { mL |= 1u << k; ++cL; }
          if (!(pv < key[l - 1 - e])) { mR |= 1u << k; ++cR; }
        }
      }
      unsigned tot;
      unsigned ex = bk::block_excl_scan<unsigned>(cL | (cR << 16), sh32, tot);     // both counts in one scan (tile <= 4096; 16 elements per thread was measured slower: 0.46 vs 0.34 ms, the strided loads stop coalescing)
      unsigned oL = nL + (ex & 0xffffu), oR = nR + (ex >> 16);
#pragma unroll
      for (int k = 0; k < IS_ITEMS; ++k) {
        if (mL & (1u << k)) scrL[lo + oL++] = lo + e0 + k;
        if (mR & (1u << k)) scrR[lo + oR++] = l - 1 - (e0 + k);
      }
      nL += tot & 0xffffu; nR += tot >> 16;
    }
    __syncthreads();
    // K = number of k with L[k] < R[k] (the predicate is true on a prefix)
    unsigned mn = min(nL, nR), kc = 0;
    for (unsigned k = threadIdx.x; k < mn; k += IS_THREADS) kc += (scrL[lo + k] < scrR[lo + k]) ? 1u : 0u;
    unsigned Ktot;
    bk::block_excl_scan<unsigned>(kc, sh32, Ktot);
    if (threadIdx.x == 0) sh_K = Ktot;
    __syncthreads();
    unsigned K = sh_K;
    for (unsigned k = threadIdx.x; k < K; k += IS_THREADS) {
      uint32_t a = scrL[lo + k], b2 = scrR[lo + k];
      uint32_t tk = key[a], tv = val[a];
      key[a] = key[b2]; val[a] = val[b2];
      key[b2] = tk; val[b2] = tv;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
      uint32_t rprev = K ? scrR[lo + K - 1] : l;
      uint32_t cut = (K < nL && scrL[lo + K] < rprev) ? scrL[lo + K] : rprev;
      seg_route(Seg{cut, l, s.depth - 1}, nxt, n_nxt, small, n_small, term, n_term);
      seg_route(Seg{f, cut, s.depth - 1}, nxt, n_nxt, small, n_small, term, n_term);
    }
    __syncthreads();
  }
}

// ---- big segments: the same partition step, one tile per CTA ---------------------------------------------------
// is_big_part   tickets hand out (segment, tile) in list order.  Tile 0 moves the median to the front and publishes the
//               pivot; every tile flags its slice from the left (L: key >= pivot) and from the right (R: key <= pivot),
//               gets "L / R entries in earlier tiles" by decoupled look-back over 64-bit status words (flag + both running
//               sums in one word) and writes its entries of the L / R position lists in place.  Earlier tiles of a segment
//               hold earlier tickets, so whatever a tile waits for is already running.
// is_big_swap   every tile finds K (the predicate L[k] < R[k] holds on a prefix: binary search), swaps its slice of the
//               K pairs; tile 0 routes the two children.
constexpr unsigned long long BS_AGG = 1ull << 62, BS_PREFIX = 2ull << 62, BS_SUM_MASK = (1ull << 31) - 1ull;

__device__ __forceinline__ const BigSeg *big_find(const BigSeg *big, unsigned nb, uint32_t ticket, unsigned &idx)
{
  unsigned a = 0, b = nb;                                    // last slot with tile_base <= ticket
  while (b - a > 1) { unsigned m = (a + b) >> 1; if (big[m].tile_base <= ticket) a = m; else b = m; }
  idx = a;
  return big + a;
}

__global__ void __launch_bounds__(IS_THREADS)
is_big_part(uint32_t *__restrict__ key, uint32_t *__restrict__ val, BigSeg *__restrict__ big, const unsigned long long *__restrict__ n_big_p,
            unsigned *__restrict__ ticket_p, unsigned long long *__restrict__ status, uint32_t *__restrict__ scrL, uint32_t *__restrict__ scrR,
            unsigned long long *__restrict__ n_big_nxt, unsigned *__restrict__ ticket_swap, Seg *__restrict__ heap, unsigned *__restrict__ n_heap)
{
  __shared__ unsigned sh32[33];
  __shared__ unsigned sh_ticket, sh_exL, sh_exR;
  const unsigned long long nbp = *n_big_p;
  const unsigned nb = (unsigned)(nbp >> 32), ntickets = (unsigned)nbp;
  if (blockIdx.x == 0 && threadIdx.x == 0) { *n_big_nxt = 0ull; *ticket_swap = 0u; }      // what is_big_swap (the next launch) counts with
  for (;;) {
    __syncthreads();
    if (threadIdx.x == 0) sh_ticket = atomicAdd(ticket_p, 1u);
    __syncthreads();
    const unsigned ticket = sh_ticket;
    if (ticket >= ntickets) return;
    unsigned si;
    const BigSeg *sp = big_find(big, nb, ticket, si);
    const uint32_t f = sp->f, l = sp->l, tile = ticket - sp->tile_base, ntiles = sp->ntiles;
    volatile BigSeg *vs = big + si;
    if (sp->depth == 0) {                                    // depth budget spent: is_heap finishes the segment
      if (tile == 0 && threadIdx.x == 0) heap[atomicAdd(n_heap, 1u)] = Seg{f, l, 0};
      continue;
    }
    if (tile == 0) {
      if (threadIdx.x == 0) {
        uint32_t mid = f + (l - f) / 2, A = f + 1, B = mid, C = l - 1;
        uint32_t ka = __ldcg(key + A), kb = __ldcg(key + B), kc = __ldcg(key + C), med;
        if (ka < kb) { if (kb < kc) med = B; else if (ka < kc) med = C; else med = A; }
        else if (ka < kc) med = A;
        else if (kb < kc) med = C;
        else med = B;
        uint32_t tk = __ldcg(key + f), tv = __ldcg(val + f), mk = __ldcg(key + med), mv = __ldcg(val + med);
        key[f] = mk; val[f] = mv; key[med] = tk; val[med] = tv;
        vs->pv = mk;
        __threadfence();
        vs->ready = 1u;
      }
    } else if (threadIdx.x == 0) {
      while (vs->ready == 0u) { }
      __threadfence();
    }
    __syncthreads();
    const uint32_t pv = vs->pv;
    const uint32_t lo = f + 1, cnt = l - lo;
    const uint32_t e0 = tile * IS_BTILE + threadIdx.x * IS_ITEMS;
    unsigned mL = 0, mR = 0, cL = 0, cR = 0;
#pragma unroll
    for (int k = 0; k < IS_ITEMS; ++k) {
      uint32_t e = e0 + k;
      if (e < cnt) {
        if (!(__ldcg(key + lo + e) < pv)) { mL |= 1u << k; ++cL; }
        if (!(pv < __ldcg(key + l - 1 - e))) { mR |= 1u << k; ++cR; }
      }
    }
    unsigned tot;
    unsigned ex = bk::block_excl_scan<unsigned>(cL | (cR << 16), sh32, tot);
    if (threadIdx.x == 0) {
      unsigned long long mine = ((unsigned long long)(tot & 0xffffu) << 31) | (unsigned long long)(tot >> 16);      // L sum << 31 | R sum
      volatile unsigned long long *st = status + ticket;
      unsigned long long exl = 0;
      if (tile == 0) *st = BS_PREFIX | mine;
      else {
        *st = BS_AGG | mine;
        for (int t = (int)ticket - 1;; --t) {
          unsigned long long sv;
          do { sv = *(volatile unsigned long long *)(status + t); } while ((sv >> 62) == 0ull);
          exl += sv & ((1ull << 62) - 1ull);
          if ((sv >> 62) == 2ull) break;
        }
        *st = BS_PREFIX | (exl + mine);
      }
      sh_exL = (unsigned)((exl >> 31) & BS_SUM_MASK); sh_exR = (unsigned)(exl & BS_SUM_MASK);
      if (tile == ntiles - 1) { vs->nL = sh_exL + (tot & 0xffffu); vs->nR = sh_exR + (tot >> 16); }
    }
    __syncthreads();
    unsigned oL = sh_exL + (ex & 0xffffu), oR = sh_exR + (ex >> 16);
#pragma unroll
    for (int k = 0; k < IS_ITEMS; ++k) {
      if (mL & (1u << k)) scrL[lo + oL++] = lo + e0 + k;
      if (mR & (1u << k)) scrR[lo + oR++] = l - 1 - (e0 + k);
    }
  }
}

__global__ void __launch_bounds__(IS_THREADS)
is_big_swap(uint32_t *__restrict__ key, uint32_t *__restrict__ val, const BigSeg *__restrict__ big, const unsigned long long *__restrict__ n_big_p,
            unsigned *__restrict__ ticket_p, const uint32_t *__restrict__ scrL, const uint32_t *__restrict__ scrR,
            Seg *__restrict__ nxt, unsigned *__restrict__ n_nxt, Seg *__restrict__ small, unsigned *__restrict__ n_small, Seg *__restrict__ term, unsigned *__restrict__ n_term,
            BigSeg *__restrict__ big_nxt, unsigned long long *__restrict__ n_big_nxt, unsigned *__restrict__ ticket_part, unsigned long long *__restrict__ status)
{
  __shared__ unsigned sh_ticket, sh_K;
  const unsigned long long nbp = *n_big_p;
  const unsigned nb = (unsigned)(nbp >> 32), ntickets = (unsigned)nbp;
  // reset what the next level's is_big_part uses: its ticket and the status words this level touched
  if (blockIdx.x == 0 && threadIdx.x == 0) *ticket_part = 0u;
  for (unsigned i = blockIdx.x * blockDim.x + threadIdx.x; i < ntickets; i += gridDim.x * blockDim.x) status[i] = 0ull;
  for (;;) {
    __syncthreads();
    if (threadIdx.x == 0) sh_ticket = atomicAdd(ticket_p, 1u);
    __syncthreads();
    const unsigned ticket = sh_ticket;
    if (ticket >= ntickets) return;
    unsigned si;
    const BigSeg *sp = big_find(big, nb, ticket, si);
    if (sp->depth == 0) continue;
    const uint32_t f = sp->f, l = sp->l, lo = f + 1, tile = ticket - sp->tile_base, nL = sp->nL, nR = sp->nR;
    const uint32_t mn = min(nL, nR);
    if (threadIdx.x == 0) {
      uint32_t a = 0, b = mn;                                // first k with !(L[k] < R[k])
      while (a < b) { uint32_t m = (a + b) >> 1; if (scrL[lo + m] < scrR[lo + m]) a = m + 1; else b = m; }
      sh_K = a;
    }
    __syncthreads();
    const uint32_t K = sh_K;
    for (uint32_t k = tile * IS_BTILE + threadIdx.x; k < K && k < (tile + 1) * IS_BTILE; k += IS_THREADS) {
      uint32_t a = scrL[lo + k], b2 = scrR[lo + k];
      uint32_t ka = __ldcg(key + a), va = __ldcg(val + a), kb = __ldcg(key + b2), vb = __ldcg(val + b2);
      key[a] = kb; val[a] = vb; key[b2] = ka; val[b2] = va;
    }
    if (tile == 0 && threadIdx.x == 0) {
      uint32_t rprev = K ? scrR[lo + K - 1] : l;
      uint32_t cut = (K < nL && scrL[lo + K] < rprev) ? scrL[lo + K] : rprev;
      seg_route(Seg{cut, l, sp->depth - 1}, nxt, n_nxt, small, n_small, term, n_term, big_nxt, n_big_nxt);
      seg_route(Seg{f, cut, sp->depth - 1}, nxt, n_nxt, small, n_small, term, n_term, big_nxt, n_big_nxt);
    }
  }
}

// Depth-exhausted segments above the small-segment size: the literal std::__partial_sort heapsort, one thread, on a copy of
// the segment in shared memory (a dependent walk down the heap per element: 30-cycle shared-memory loads instead of L2 round
// trips).  Near-sorted input -- the p2 order of a same-chromosome bucket right after its p1 sort -- drives median-of-3 into
// its worst case, so deep-coverage buckets DO end here: a 4 459 element segment took ~10 ms from global memory.
constexpr uint32_t IS_HEAP_SMEM_ELEMS = 25600;          // 200 KB of (key, value)

// the same heapsort as seg_heapsort on (key, value) pairs held as one 8-byte word each, 32-bit indices; H[1] is 16-byte
// aligned, so the two children of a hole (indices 2h+1, 2h+2) come with ONE 16-byte load
__device__ __forceinline__ void heap_adjust_pairs(uint2 *H, int hole, int len, uint2 v)
{
  const int top = hole;
  int child = hole;
  const int lim = (len - 1) / 2;
  while (child < lim) {
    child = 2 * (child + 1);
    uint4 c2 = *reinterpret_cast<const uint4 *>(H + child - 1);          // (key, val) of child-1 and of child
    uint2 pick = make_uint2(c2.z, c2.w);
    if (c2.z < c2.x) { --child; pick = make_uint2(c2.x, c2.y); }
    H[hole] = pick;
    hole = child;
  }
  if ((len & 1) == 0 && child == (len - 2) / 2) {
    child = 2 * (child + 1);
    H[hole] = H[child - 1];
    hole = child - 1;
  }
  int parent = (hole - 1) / 2;
  while (hole > top && H[parent].x < v.x) {
    H[hole] = H[parent];
    hole = parent;
    parent = (hole - 1) / 2;
  }
  H[hole] = v;
}
__device__ __forceinline__ void heapsort_pairs(uint2 *H, int n)
{
  if (n < 2) return;
  for (int parent = (n - 2) / 2;; --parent) {
    heap_adjust_pairs(H, parent, n, H[parent]);
    if (parent == 0) break;
  }
  for (int last = n - 1; last > 0; --last) {
    uint2 v = H[last];
    H[last] = H[0];
    heap_adjust_pairs(H, 0, last, v);
  }
}

__global__ void __launch_bounds__(256) is_heap(uint32_t *__restrict__ key, uint32_t *__restrict__ val, const Seg *__restrict__ heap, const unsigned *__restrict__ n_heap_p)
{
  extern __shared__ __align__(16) unsigned char hs_raw[];
  uint2 *H = reinterpret_cast<uint2 *>(hs_raw + 8);        // &H[1] is 16-byte aligned
  const unsigned n_heap = *n_heap_p;
  for (unsigned si = blockIdx.x; si < n_heap; si += gridDim.x) {
    const uint32_t f = heap[si].f, l = heap[si].l, n = l - f;
    if (n > IS_HEAP_SMEM_ELEMS) {
      if (threadIdx.x == 0) seg_heapsort(key, val, f, l);
      continue;
    }
    __syncthreads();
    for (uint32_t i = threadIdx.x; i < n; i += blockDim.x) H[i] = make_uint2(key[f + i], val[f + i]);
    __syncthreads();
    if (threadIdx.x == 0) heapsort_pairs(H, (int)n);
    __syncthreads();
    for (uint32_t i = threadIdx.x; i < n; i += blockDim.x) { uint2 e = H[i]; key[f + i] = e.x; val[f + i] = e.y; }
  }
}

__global__ void is_terminal(uint32_t *__restrict__ key, uint32_t *__restrict__ val, const Seg *__restrict__ term, const unsigned *__restrict__ n_term)
{
  unsigned t = blockIdx.x * blockDim.x + threadIdx.x;
  unsigned n = *n_term;
  for (; t < n; t += gridDim.x * blockDim.x) seg_insertion_sort(key, val, term[t].f, term[t].l);
}

// =============================================================================================
// K4: isolated-pair mask (src/BreakID.cc:1813-1877) over all buckets at once.
// cur[] holds pair ids in the current (sorted) order, seg_off the bucket boundaries.
// out_count[p] = how many copies of element p survive (0, 1, or 2 for position 1 of a bucket).
// =============================================================================================
__device__ __forceinline__ long long gap32(uint32_t a, uint32_t b)
{
  int32_t d = (int32_t)(a - b);
  return d < 0 ? -(long long)d : (long long)d;
}

__global__ void k4_mask_count(const uint32_t *__restrict__ cur, const uint32_t *__restrict__ bucket_of, const uint32_t *__restrict__ seg_off,
                              long long np, const uint32_t *__restrict__ x, const uint32_t *__restrict__ y, long long distance,
                              uint32_t *__restrict__ out_count)
{
  long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= np) return;
  uint32_t b = bucket_of[p];
  uint32_t s = seg_off[b], e = seg_off[b + 1];
  uint32_t n = e - s, i = (uint32_t)p - s;
  unsigned c = 0;
  if (n >= 3 && i >= 1 && i + 1 < n) {
    uint32_t a = cur[p - 1], m = cur[p], z = cur[p + 1];
    long long ll = gap32(x[a], x[m]), lr = gap32(x[z], x[m]);
    long long Lx = ll < lr ? ll : lr;
    ll = gap32(y[a], y[m]); lr = gap32(y[z], y[m]);
    long long Ly = ll < lr ? ll : lr;
    if (!(Lx > distance || Ly > distance)) c = 1;
    if (i == 1) {                                            // "first read pair" test uses e[1], e[2] (:1830-1835)
      long long fx = gap32(x[m], x[z]), fy = gap32(y[m], y[z]);
      if (!(fx > distance || fy > distance)) c += 1;
    }
  }
  out_count[p] = c;
}

__global__ void k4_mask_write(const uint32_t *__restrict__ cur, const uint32_t *__restrict__ bucket_of, long long np,
                              const uint32_t *__restrict__ out_count, const uint32_t *__restrict__ out_off,
                              uint32_t *__restrict__ cur_out, uint32_t *__restrict__ bucket_of_out)
{
  long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= np) return;
  uint32_t c = out_count[p], o = out_off[p];
  for (uint32_t k = 0; k < c; ++k) { cur_out[o + k] = cur[p]; bucket_of_out[o + k] = bucket_of[p]; }
}

// new bucket offsets = scanned offsets sampled at the old bucket starts
__global__ void k4_new_offsets(const uint32_t *__restrict__ seg_off, int nb, const uint32_t *__restrict__ out_off, long long np, unsigned long long total,
                               uint32_t *__restrict__ seg_off_out)
{
  int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b > nb) return;
  uint32_t s = seg_off[b];
  seg_off_out[b] = (s < np) ? out_off[s] : (uint32_t)total;
}

__global__ void gather_u32(const uint32_t *__restrict__ src, const uint32_t *__restrict__ idx, long long n, uint32_t *__restrict__ dst)
{
  long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (p < n) dst[p] = src[idx[p]];
}
__global__ void iota_u32(uint32_t *dst, long long n)
{
  long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (p < n) dst[p] = (uint32_t)p;
}
__global__ void pair_xy(const bkid_pair *__restrict__ pairs, long long np, uint32_t *__restrict__ x, uint32_t *__restrict__ y, uint32_t *__restrict__ bucket_of)
{
  long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (p < np) { x[p] = pairs[p].p1_chr_pos; y[p] = pairs[p].p2_chr_pos; bucket_of[p] = (uint32_t)pairs[p].bucket; }
}

#include "bkid_cluster.cuh"
#include "bkid_refine.cuh"
#include "bkid_align.cuh"
#include "bkid_api.cuh"
#include "bkid_sort.cuh"
#include "bkid_dist.cuh"
#include "bkid_bamdec.cuh"
#include "bkid_samdec.cuh"
#include "bkid_align_api.cuh"
