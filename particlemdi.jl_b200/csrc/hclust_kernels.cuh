// Exact agglomerative clustering of the pooled pair counts (pmdi_summary_hclust, include/pmdi_cuda.h; DESIGN.md §16):
// single, complete and average linkage on the similarity numerators A_ij of a summary.  Shares no device code with
// the sweep engines; reads the counts in the layout of summary_kernels.cuh.
//
// Working state.  W is the full n x n square of cluster similarities s(X, Y) between active clusters, indexed by
// their representatives (smallest observation index): uint32 for single / complete (a max or min of A_ij <= 2^27),
// uint64 for average (a sum, < 2^57).  Every active row i caches its best partner (value, p, column), the smallest
// column among equals.  A pair's value is s / p with p = |X||Y| for average and 1 otherwise; values are compared
// exactly as s1 p2 against s2 p1 in 128 bits, and equal values go to the lexicographically smallest (smaller rep,
// larger rep).  Then the best pair of all is the best among the row caches: row a of the best pair (a, b) caches b.
#pragma once
#include <climits>
#include <cstdint>

#include "summary_kernels.cuh"

namespace hclust {

enum { LINK_SINGLE = 0, LINK_COMPLETE = 1, LINK_AVERAGE = 2 };
constexpr int HC_THREADS = 512;
constexpr int HC_ERR_WATCHDOG = 77;  // a grid barrier waited longer than the watchdog allows
constexpr int HC_ERR_PAIR = 78;      // no valid best pair (cannot happen while two clusters are active)

struct HcKey {
  unsigned long long s, p;
  int lo, hi;  // the pair (lo < hi), or in a row scan the column twice
};

struct HcMerge {
  int a, b;         // representatives, a < b; the merged cluster keeps a
  unsigned size;    // |a| + |b|
  unsigned p;       // 1, or |a| |b| for average
  unsigned long long s;
};

struct HcArgs {
  void* W;                  // [n][n] of the linkage's value type
  unsigned* size;           // cluster size per representative, 0 once retired
  unsigned long long* cs;   // row caches: value, p and column of every row's best partner
  unsigned* cp;
  int* cj;
  int* list;                // rows to rescan in this merge
  unsigned* cnt;            // [2] list lengths, by merge parity
  HcKey* part;              // [2 parities][2 phases][G] per-CTA best pairs
  HcKey* rowa;              // [G] per-CTA best entry of the merged row
  HcMerge* rec;             // [n - 1]
  unsigned long long* bar;  // grid barrier counter (zeroed before the launch)
  int* err;
  unsigned long long* rescans;
  int n;
  unsigned long long wd_ns;
};

__device__ __forceinline__ HcKey hc_empty() { return HcKey{0ull, 1ull, INT_MAX, INT_MAX}; }

// x better than y: a larger s / p, or an equal one with a smaller (lo, hi); exact (s < 2^57, p < 2^30)
__device__ __forceinline__ bool hc_better(const HcKey& x, const HcKey& y) {
  const unsigned long long xh = __umul64hi(x.s, y.p), yh = __umul64hi(y.s, x.p);
  if (xh != yh) return xh > yh;
  const unsigned long long xl = x.s * y.p, yl = y.s * x.p;
  if (xl != yl) return xl > yl;
  return x.lo < y.lo || (x.lo == y.lo && x.hi < y.hi);
}

__device__ __forceinline__ HcKey hc_shfl(const HcKey& v, int o) {
  return HcKey{__shfl_xor_sync(0xffffffffu, v.s, o), __shfl_xor_sync(0xffffffffu, v.p, o),
               __shfl_xor_sync(0xffffffffu, v.lo, o), __shfl_xor_sync(0xffffffffu, v.hi, o)};
}

// the best of the CTA's keys, returned to every thread; sh holds a key per warp
__device__ __forceinline__ HcKey hc_block_best(HcKey v, HcKey* sh) {
#pragma unroll
  for (int o = 16; o; o >>= 1) {
    const HcKey w = hc_shfl(v, o);
    if (hc_better(w, v)) v = w;
  }
  if (threadIdx.x % 32 == 0) sh[threadIdx.x / 32] = v;
  __syncthreads();
  v = sh[0];
  for (int w = 1; w < (int)blockDim.x / 32; ++w)
    if (hc_better(sh[w], v)) v = sh[w];
  __syncthreads();
  return v;
}

// the row-cache entry (value, p, column j) of row i as the pair key of (i, j)
__device__ __forceinline__ HcKey hc_pair(const HcKey& r, int i) {
  return r.lo == INT_MAX ? r : HcKey{r.s, r.p, min(i, r.lo), max(i, r.lo)};
}

// Best partner of row i over the active columns, by the whole CTA.  During merge (a, b) the sizes of a and b are
// taken as (snew, 0), whatever the size array holds while CTA 0 updates it; a = b = -1 outside a merge.
template <int LINK, class V>
__device__ __forceinline__ HcKey hc_scan_row(const V* W, const unsigned* size, int n, int i, int a, int b,
                                             unsigned snew, HcKey* sh) {
  HcKey best = hc_empty();
  const V* row = W + (size_t)i * n;
  const unsigned si = i == a ? snew : size[i];
  for (int j = threadIdx.x; j < n; j += blockDim.x) {
    const unsigned sj = j == a ? snew : j == b ? 0u : size[j];
    if (j == i || !sj) continue;
    const HcKey c{(unsigned long long)row[j], LINK == LINK_AVERAGE ? (unsigned long long)si * sj : 1ull, j, j};
    if (hc_better(c, best)) best = c;
  }
  return hc_block_best(best, sh);
}

__device__ __forceinline__ unsigned long long hc_now_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
  return t;
}
__device__ __forceinline__ unsigned long long hc_ld_acquire(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}

// grid barrier of the merge kernel, all threads; false (error set) when it waited longer than wd_ns or another CTA
// failed, so that every CTA leaves instead of spinning forever
__device__ __forceinline__ bool hc_gsync(const HcArgs& g, unsigned long long& epoch, int& fail) {
  __syncthreads();
  if (threadIdx.x == 0) {
    epoch += gridDim.x;
    __threadfence();
    atomicAdd(g.bar, 1ull);
    if (hc_ld_acquire(g.bar) < epoch) {
      const unsigned long long t0 = hc_now_ns();
      unsigned spins = 0;
      while (hc_ld_acquire(g.bar) < epoch) {
        if (((++spins) & 0x3ffu) == 0) {
          if (__ldcg(g.err) != 0) { fail = 1; break; }
          if (hc_now_ns() - t0 > g.wd_ns) { atomicExch(g.err, HC_ERR_WATCHDOG); fail = 1; break; }
        }
      }
    }
  }
  __syncthreads();
  return fail == 0;
}

// W[i][j] = A_ij of the pooled chains c0..c1-1, for dataset k or summed over the K datasets (k < 0); mirrored from the
// upper-triangle tiles, 0 on the diagonal.  A 32 x 32 block per CTA of 32 x 8 threads; blocks below the diagonal read
// the mirror block coalesced and transpose it in shared memory (as k_summary_psm).
template <class V>
__global__ void __launch_bounds__(256) k_hclust_fill(const unsigned* counts, int C, size_t chain_stride,
                                                     size_t k_stride, int K, int k, int T, long long n, V* W) {
  __shared__ V sm[32][33];
  const long long bi = (long long)blockIdx.y * 32, bj = (long long)blockIdx.x * 32;
  const int tx = threadIdx.x % 32, ty = threadIdx.x / 32;
  auto A = [&](long long a, long long b) -> V {  // a <= b
    if (a == b) return (V)0;
    if (k >= 0) return (V)summary::sum_count(counts, 0, C, chain_stride, (size_t)k * k_stride, T, a, b);
    unsigned long long s = 0;
    for (int q = 0; q < K; ++q) s += summary::sum_count(counts, 0, C, chain_stride, (size_t)q * k_stride, T, a, b);
    return (V)s;
  };
  if (bi > bj) {
#pragma unroll
    for (int m = 0; m < 4; ++m) {
      const long long a = bj + ty + 8 * m, b = bi + tx;  // a < b
      if (a < n && b < n) sm[ty + 8 * m][tx] = A(a, b);
    }
    __syncthreads();
#pragma unroll
    for (int m = 0; m < 4; ++m) {
      const long long i = bi + ty + 8 * m, j = bj + tx;
      if (i < n && j < n) W[i * n + j] = sm[tx][ty + 8 * m];
    }
  } else {
#pragma unroll
    for (int m = 0; m < 4; ++m) {
      const long long i = bi + ty + 8 * m, j = bj + tx;
      if (i < n && j < n) W[i * n + j] = A(i < j ? i : j, i < j ? j : i);
    }
  }
}

// All n - 1 merges in one cooperative launch.  First every row's cache is filled by a row scan (a CTA per row).  Then
// each merge m, with two grid barriers:
//   pick   every CTA reduces the per-CTA best pairs of the previous merge to the same (a, b);
//   A      a thread per observation j: W[a][j] = W[j][a] = max / min / sum of W[a][j] and W[b][j]; a row whose cache
//          is a or b goes on the rescan list (single linkage never needs one: the new entry in column a is then the
//          row's maximum and a its smallest column); every other row compares its new entry in column a against its
//          cache.  The merged row's own best is reduced from the same entries, a per-CTA partial;
//   B      CTA 0 takes row a's best from those partials and updates the sizes; the CTAs rescan the listed rows.
// Per-CTA best pairs of A and B feed the next pick, through buffers alternating by merge parity.
template <int LINK, class V>
__global__ void __launch_bounds__(HC_THREADS) k_hclust_merge(HcArgs g) {
  __shared__ HcKey sh[HC_THREADS / 32];
  __shared__ unsigned long long epoch;
  __shared__ int fail;
  if (threadIdx.x == 0) { epoch = 0; fail = 0; }
  __syncthreads();
  V* W = (V*)g.W;
  const int n = g.n, G = gridDim.x;
  HcKey best = hc_empty();
  for (int i = blockIdx.x; i < n; i += G) {
    const HcKey r = hc_scan_row<LINK>(W, g.size, n, i, -1, -1, 0u, sh);
    if (threadIdx.x == 0) { g.cs[i] = r.s; g.cp[i] = (unsigned)r.p; g.cj[i] = r.lo; }
    const HcKey c = hc_pair(r, i);
    if (hc_better(c, best)) best = c;
  }
  if (threadIdx.x == 0) { g.part[blockIdx.x] = hc_empty(); g.part[G + blockIdx.x] = best; }
  if (!hc_gsync(g, epoch, fail)) return;
  unsigned long long rescans = 0;
  for (int m = 0; m < n - 1; ++m) {
    const HcKey* in = g.part + (size_t)(m & 1) * 2 * G;
    HcKey* out = g.part + (size_t)((m + 1) & 1) * 2 * G;
    HcKey w = hc_empty();
    for (int e = threadIdx.x; e < 2 * G; e += blockDim.x)
      if (hc_better(in[e], w)) w = in[e];
    w = hc_block_best(w, sh);
    const int a = w.lo, b = w.hi;
    if (a < 0 || a >= b || b >= n) {  // the same on every CTA: all leave together
      if (blockIdx.x == 0 && threadIdx.x == 0) atomicExch(g.err, HC_ERR_PAIR);
      return;
    }
    const unsigned snew = g.size[a] + g.size[b];
    if (blockIdx.x == 0 && threadIdx.x == 0) g.rec[m] = HcMerge{a, b, snew, (unsigned)w.p, w.s};
    unsigned* cnt = g.cnt + (m & 1);
    const V* ra = W + (size_t)a * n;
    const V* rb = W + (size_t)b * n;
    HcKey bestA = hc_empty(), rowa = hc_empty();
    for (int base = blockIdx.x * blockDim.x; base < n; base += G * blockDim.x) {
      const int j = base + threadIdx.x;
      bool push = false;
      if (j < n && j != a && j != b && g.size[j]) {
        const V va = ra[j], vb = rb[j];
        const V v = LINK == LINK_SINGLE ? (va > vb ? va : vb) : LINK == LINK_COMPLETE ? (va < vb ? va : vb) : va + vb;
        W[(size_t)a * n + j] = v;
        W[(size_t)j * n + a] = v;
        const unsigned long long p = LINK == LINK_AVERAGE ? (unsigned long long)snew * g.size[j] : 1ull;
        const HcKey e{(unsigned long long)v, p, j, j};
        if (hc_better(e, rowa)) rowa = e;
        int c = g.cj[j];
        HcKey cur{g.cs[j], g.cp[j], c, c};
        const HcKey na{(unsigned long long)v, p, a, a};
        if (LINK == LINK_SINGLE && (c == a || c == b)) {
          cur = na;
        } else if (c == a || c == b) {
          push = true;
        } else if (hc_better(na, cur)) {
          cur = na;
        }
        if (!push) {
          if (cur.lo != c) { g.cs[j] = cur.s; g.cp[j] = (unsigned)cur.p; g.cj[j] = cur.lo; }
          const HcKey pk = hc_pair(cur, j);
          if (hc_better(pk, bestA)) bestA = pk;
        }
      }
      const unsigned ball = __ballot_sync(0xffffffffu, push);
      if (ball) {
        const int lane = threadIdx.x % 32;
        unsigned at = 0;
        if (lane == __ffs(ball) - 1) at = atomicAdd(cnt, (unsigned)__popc(ball));
        at = __shfl_sync(0xffffffffu, at, __ffs(ball) - 1);
        if (push) g.list[at + __popc(ball & ((1u << lane) - 1u))] = j;
      }
    }
    bestA = hc_block_best(bestA, sh);
    rowa = hc_block_best(rowa, sh);
    if (threadIdx.x == 0) { out[blockIdx.x] = bestA; g.rowa[blockIdx.x] = rowa; }
    if (!hc_gsync(g, epoch, fail)) return;
    HcKey bestB = hc_empty();
    if (blockIdx.x == 0) {
      HcKey r = hc_empty();
      for (int e = threadIdx.x; e < G; e += blockDim.x)
        if (hc_better(g.rowa[e], r)) r = g.rowa[e];
      r = hc_block_best(r, sh);
      if (threadIdx.x == 0) {
        g.cs[a] = r.s; g.cp[a] = (unsigned)r.p; g.cj[a] = r.lo;
        g.size[a] = snew;
        g.size[b] = 0;
        g.cnt[(m + 1) & 1] = 0;  // last read in merge m - 1's phase B
      }
      bestB = hc_pair(r, a);
    }
    const unsigned L = __ldcg(cnt);
    rescans += L;
    for (unsigned e = blockIdx.x; e < L; e += G) {
      const int i = __ldcg(g.list + e);
      const HcKey r = hc_scan_row<LINK>(W, g.size, n, i, a, b, snew, sh);
      if (threadIdx.x == 0) { g.cs[i] = r.s; g.cp[i] = (unsigned)r.p; g.cj[i] = r.lo; }
      const HcKey c = hc_pair(r, i);
      if (hc_better(c, bestB)) bestB = c;
    }
    if (threadIdx.x == 0) out[G + blockIdx.x] = bestB;
    if (!hc_gsync(g, epoch, fail)) return;
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) *g.rescans = rescans;
}

}  // namespace hclust
