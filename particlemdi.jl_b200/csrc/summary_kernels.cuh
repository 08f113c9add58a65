// Posterior summaries of retained allocations (pmdi_summary_*, include/pmdi_cuda.h; DESIGN.md §14): pair agreement
// counts, posterior similarity read-out, least-squares consensus losses and cross-chain agreement.  Shares no device
// code with the sweep engines.
//
// Layout.  Labels are stored as uint8 (label - 1) in chunks of SUM_CH samples of one chain, [k][i][r]: the SUM_CH
// samples of observation i of dataset k are adjacent, so four consecutive samples are one 32-bit word.  Counts are
// uint32, upper triangle only, in SUM_TILE x SUM_TILE tiles (ti <= tj, row-major over the triangle; a diagonal tile is
// stored whole), [chain][k][tile][il][jl].
#pragma once
#include <cstdint>

namespace summary {

constexpr int SUM_TILE = 128;      // observations per tile side
constexpr int SUM_CH = 256;        // samples per chunk (a chunk of one chain is counted in one pass)
constexpr int SUM_SW = 16;         // words (4 samples each) staged in shared memory per step
constexpr int SUM_THREADS = 256;   // 16 x 16 threads, each with an 8 x 8 block of pairs
constexpr int SUM_TE = SUM_TILE * SUM_TILE;
constexpr int SUM_MAX_JOBS = 64;   // chains counted in one launch
constexpr int SUM_LS_CHUNKS = 12;  // chunks (3,072 samples) per launch of the least-squares pass
// the word walks start at multiples of SUM_SW and stop before word ceil(r1 / 4) <= SUM_CH / 4: whole steps of SUM_SW
// words then end exactly at the end of an observation's row
static_assert((SUM_CH / 4) % SUM_SW == 0, "an observation's row is a whole number of staging steps");

struct CountJob {
  const uint8_t* chunk;  // [k][i][SUM_CH]
  unsigned* counts;      // the chain's counts, [k][tile][SUM_TE]
  int r0, r1;            // samples r0 <= r < r1 of the chunk
};
struct CountJobs { CountJob j[SUM_MAX_JOBS]; };

struct LsBatch {
  const uint8_t* chunk[SUM_LS_CHUNKS];
  int r1[SUM_LS_CHUNKS];    // samples 0 <= r < r1 of each chunk
  int base[SUM_LS_CHUNKS];  // index of the chunk's first sample among the launch's samples
  int n_chunks, n_samples;
};

// tile t of the upper triangle of T x T tiles -> (ti, tj), ti <= tj
__device__ __forceinline__ void sum_tile_of(int t, int T, int& ti, int& tj) {
  ti = 0;
  while (t >= T - ti) { t -= T - ti; ++ti; }
  tj = ti + t;
}

// 0x80 in every byte where a and b agree, 0 elsewhere
__device__ __forceinline__ unsigned sum_eq80(unsigned a, unsigned b) {
  const unsigned x = a ^ b;
  const unsigned t = (x & 0x7f7f7f7fu) + 0x7f7f7f7fu;
  return ~(t | x) & 0x80808080u;
}

// Stage SUM_SW words (from word w0 of the chunk) of the 128 observations from `base`: s[w][o].  Bytes of samples
// outside [r0, r1) become 0x00 on the i side and 0xff on the j side, so they never agree; observations past n, and
// words past the end of an observation's SUM_CH bytes, read 0.  Callers start w0 at a multiple of SUM_SW, so with
// r1 <= SUM_CH every staged word lies inside the row anyway; the guard keeps a read inside the chunk allocation
// whatever the caller passes.
__device__ __forceinline__ void sum_stage(unsigned (*si)[SUM_TILE + 4], unsigned (*sj)[SUM_TILE + 4],
                                          const uint8_t* lab, long long n, long long bi, long long bj, int w0, int r0,
                                          int r1) {
  const int w = threadIdx.x % SUM_SW;
  const bool in_row = w0 + w < SUM_CH / 4;
  const int lo = r0 - 4 * (w0 + w), hi = r1 - 4 * (w0 + w);
  unsigned m = 0;
#pragma unroll
  for (int b = 0; b < 4; ++b)
    if (b >= lo && b < hi) m |= 0xffu << (8 * b);
#pragma unroll
  for (int q = 0; q < SUM_TILE * SUM_SW / SUM_THREADS; ++q) {
    const int o = threadIdx.x / SUM_SW + q * (SUM_THREADS / SUM_SW);
    const long long i = bi + o, j = bj + o;
    const unsigned vi = in_row && i < n ? reinterpret_cast<const unsigned*>(lab + (size_t)i * SUM_CH)[w0 + w] : 0u;
    const unsigned vj = in_row && j < n ? reinterpret_cast<const unsigned*>(lab + (size_t)j * SUM_CH)[w0 + w] : 0u;
    si[w][o] = vi & m;
    sj[w][o] = vj | ~m;
  }
}

// the 8 observations of a thread on one side: 4t..4t+3 and 64+4t..64+4t+3
__device__ __forceinline__ int sum_local(int t, int x) { return (x < 4 ? 4 * t : 60 + 4 * t) + x; }

__device__ __forceinline__ void sum_load8(const unsigned* row, int t, unsigned (&v)[8]) {
  const uint4 a = *reinterpret_cast<const uint4*>(row + 4 * t);
  const uint4 b = *reinterpret_cast<const uint4*>(row + 64 + 4 * t);
  v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
}

// count[chain][k][i][j] += samples r0 <= r < r1 of the job's chunk in which i and j agree.  grid (tiles, K, jobs).
__global__ void __launch_bounds__(SUM_THREADS) k_summary_count(CountJobs jobs, long long n, int T, int tiles) {
  __shared__ __align__(16) unsigned si[SUM_SW][SUM_TILE + 4];
  __shared__ __align__(16) unsigned sj[SUM_SW][SUM_TILE + 4];
  const CountJob job = jobs.j[blockIdx.z];
  const int k = blockIdx.y;
  int ti, tj;
  sum_tile_of(blockIdx.x, T, ti, tj);
  const uint8_t* lab = job.chunk + (size_t)k * n * SUM_CH;
  const int tx = threadIdx.x % 16, ty = threadIdx.x / 16;
  // 0x80 per agreeing sample: at most SUM_CH * 0x80 = 2^15 per pass, folded into the uint32 counts at the end
  unsigned acc[8][8];
#pragma unroll
  for (int x = 0; x < 8; ++x)
#pragma unroll
    for (int y = 0; y < 8; ++y) acc[x][y] = 0;
  // from the staging step that holds sample r0 (samples below r0 in it are masked): the last step ends at word
  // SUM_CH / 4 at most
  for (int w0 = job.r0 / 4 / SUM_SW * SUM_SW; w0 < (job.r1 + 3) / 4; w0 += SUM_SW) {
    __syncthreads();
    sum_stage(si, sj, lab, n, (long long)ti * SUM_TILE, (long long)tj * SUM_TILE, w0, job.r0, job.r1);
    __syncthreads();
#pragma unroll 1
    for (int w = 0; w < SUM_SW; ++w) {
      unsigned a[8], b[8];
      sum_load8(si[w], ty, a);
      sum_load8(sj[w], tx, b);
#pragma unroll
      for (int x = 0; x < 8; ++x)
#pragma unroll
        for (int y = 0; y < 8; ++y) acc[x][y] = __dp4a(sum_eq80(a[x], b[y]), 0x01010101u, acc[x][y]);
    }
  }
  unsigned* cnt = job.counts + ((size_t)k * tiles + blockIdx.x) * SUM_TE;
#pragma unroll
  for (int x = 0; x < 8; ++x) {
    unsigned* row = cnt + sum_local(ty, x) * SUM_TILE;
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      uint4* p = reinterpret_cast<uint4*>(row + 64 * h + 4 * tx);
      uint4 c = *p;
      c.x += acc[x][4 * h] >> 7; c.y += acc[x][4 * h + 1] >> 7; c.z += acc[x][4 * h + 2] >> 7; c.w += acc[x][4 * h + 3] >> 7;
      *p = c;
    }
  }
}

// one added sample: in[k][i] -> chunk[k][i][r]
__global__ void k_summary_put(const uint8_t* in, uint8_t* chunk, long long total, int r) {
  for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x)
    chunk[e * SUM_CH + r] = in[e];
}

// sample r of a chunk, dataset k -> out[i] (labels - 1)
__global__ void k_summary_get(const uint8_t* chunk, uint8_t* out, long long n, int r) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    out[i] = chunk[i * SUM_CH + r];
}

// count of pair (a <= b)
__device__ __forceinline__ unsigned long long sum_count(const unsigned* counts, int c0, int c1, size_t chain_stride,
                                                        size_t k_off, int T, long long a, long long b) {
  const int ti = (int)(a / SUM_TILE), tj = (int)(b / SUM_TILE);
  const size_t t = (size_t)ti * T - (size_t)ti * (ti - 1) / 2 + (tj - ti);
  const size_t e = k_off + t * SUM_TE + (a % SUM_TILE) * SUM_TILE + (b % SUM_TILE);
  unsigned long long s = 0;
  for (int c = c0; c < c1; ++c) s += counts[c * chain_stride + e];
  return s;
}

// PSM of pair (a <= b): chains c0..c1-1 pooled, dataset k, or the mean over the K datasets in k order (k < 0)
__device__ __forceinline__ double sum_psm(const unsigned* counts, int c0, int c1, size_t chain_stride, size_t k_stride,
                                          int K, int k, int T, double rows, long long a, long long b) {
  if (k >= 0) return (double)sum_count(counts, c0, c1, chain_stride, k * k_stride, T, a, b) / rows;
  double acc = 0.0;
  for (int q = 0; q < K; ++q) acc += (double)sum_count(counts, c0, c1, chain_stride, q * k_stride, T, a, b) / rows;
  return acc / (double)K;
}

// the full n x n PSM, mirrored; a 32 x 32 block per CTA of 32 x 8 threads (blocks below the diagonal read the mirror
// block coalesced and transpose it in shared memory)
template <class O>
__global__ void __launch_bounds__(256) k_summary_psm(const unsigned* counts, int c0, int c1, size_t chain_stride,
                                                     size_t k_stride, int K, int k, int T, double rows, long long n,
                                                     O* out) {
  __shared__ double sm[32][33];
  const long long bi = (long long)blockIdx.y * 32, bj = (long long)blockIdx.x * 32;
  const int tx = threadIdx.x % 32, ty = threadIdx.x / 32;
  if (bi > bj) {
#pragma unroll
    for (int m = 0; m < 4; ++m) {
      const long long a = bj + ty + 8 * m, b = bi + tx;  // a < b
      if (a < n && b < n) sm[ty + 8 * m][tx] = sum_psm(counts, c0, c1, chain_stride, k_stride, K, k, T, rows, a, b);
    }
    __syncthreads();
#pragma unroll
    for (int m = 0; m < 4; ++m) {
      const long long i = bi + ty + 8 * m, j = bj + tx;
      if (i < n && j < n) out[i * n + j] = (O)sm[tx][ty + 8 * m];
    }
  } else {
#pragma unroll
    for (int m = 0; m < 4; ++m) {
      const long long i = bi + ty + 8 * m, j = bj + tx;
      if (i < n && j < n)
        out[i * n + j] = (O)sum_psm(counts, c0, c1, chain_stride, k_stride, K, k, T, rows, i < j ? i : j, i < j ? j : i);
    }
  }
}

// Least-squares losses of one batch of samples of dataset k against the pooled counts.  With R the pooled rows and
// w_ij = R - 2 count_ij, R^2 L_r = R * T_r + Q where T_r = sum_{i<j, s_i = s_j} w_ij and Q = sum_{i<j} count_ij^2
// (both exact integers; Q in 128 bits, q[0] low and q[1] high word).  Each CTA walks tiles blockIdx.x, +gridDim.x, ...; per-sample sums are exact, so the order
// in which they are added does not matter.  tsum[sample] and q[0..1] (when want_q) are zeroed by the caller.
__global__ void __launch_bounds__(SUM_THREADS) k_summary_ls(LsBatch batch, const unsigned* counts, int C,
                                                            size_t chain_stride, size_t k_off, long long n, int T,
                                                            int tiles, long long R, unsigned long long* tsum,
                                                            unsigned long long* q, int want_q) {
  __shared__ __align__(16) unsigned si[SUM_SW][SUM_TILE + 4];
  __shared__ __align__(16) unsigned sj[SUM_SW][SUM_TILE + 4];
  __shared__ unsigned long long part[SUM_LS_CHUNKS * SUM_CH];
  for (int s = threadIdx.x; s < batch.n_samples; s += SUM_THREADS) part[s] = 0;
  const int tx = threadIdx.x % 16, ty = threadIdx.x / 16, lane = threadIdx.x % 32;
  for (int t = blockIdx.x; t < tiles; t += gridDim.x) {
    int ti, tj;
    sum_tile_of(t, T, ti, tj);
    int wgt[8][8];
    unsigned long long qtile = 0;  // <= 64 pairs x (2^24)^2 = 2^54 per thread, 2^59 per warp
#pragma unroll
    for (int x = 0; x < 8; ++x) {
      const long long i = (long long)ti * SUM_TILE + sum_local(ty, x);
#pragma unroll
      for (int y = 0; y < 8; ++y) {
        const long long j = (long long)tj * SUM_TILE + sum_local(tx, y);
        unsigned long long c = 0;
        if (i < j && j < n) {
          const size_t e = k_off + (size_t)t * SUM_TE + (size_t)sum_local(ty, x) * SUM_TILE + sum_local(tx, y);
          for (int ch = 0; ch < C; ++ch) c += counts[ch * chain_stride + e];
          qtile += c * c;
          wgt[x][y] = (int)(R - 2 * (long long)c);
        } else {
          wgt[x][y] = 0;
        }
      }
    }
    if (want_q) {  // Q can exceed 2^64 (n_obs^2 / 2 pairs x R^2): a 128-bit sum, low word with its carries in q[1]
      for (int o = 16; o; o >>= 1) qtile += __shfl_xor_sync(0xffffffffu, qtile, o);
      if (lane == 0 && qtile && atomicAdd(&q[0], qtile) + qtile < qtile) atomicAdd(&q[1], 1ull);
    }
    for (int ck = 0; ck < batch.n_chunks; ++ck) {
      const uint8_t* labk = batch.chunk[ck];  // dataset k of the chunk
      const int r1 = batch.r1[ck];
      for (int w0 = 0; w0 < (r1 + 3) / 4; w0 += SUM_SW) {
        __syncthreads();
        sum_stage(si, sj, labk, n, (long long)ti * SUM_TILE, (long long)tj * SUM_TILE, w0, 0, r1);
        __syncthreads();
        for (int w = 0; w < SUM_SW && 4 * (w0 + w) < r1; ++w) {
          unsigned a[8], b[8];
          sum_load8(si[w], ty, a);
          sum_load8(sj[w], tx, b);
          int s0 = 0, s1 = 0, s2 = 0, s3 = 0;  // |s| <= 64 R < 2^31 (R <= 2^24)
#pragma unroll
          for (int x = 0; x < 8; ++x)
#pragma unroll
            for (int y = 0; y < 8; ++y) {
              const unsigned z = sum_eq80(a[x], b[y]);
              const int v = wgt[x][y];
              s0 += (int)((z >> 7) & 1u) * v;
              s1 += (int)((z >> 15) & 1u) * v;
              s2 += (int)((z >> 23) & 1u) * v;
              s3 += (int)(z >> 31) * v;
            }
          int sv[4] = {s0, s1, s2, s3};
#pragma unroll
          for (int b4 = 0; b4 < 4; ++b4) {
            // exact warp sum of 32 values |v| < 2^31: low 16 bits and the rest summed apart
            const unsigned lo = __reduce_add_sync(0xffffffffu, (unsigned)sv[b4] & 0xffffu);
            const int hi = __reduce_add_sync(0xffffffffu, sv[b4] >> 16);
            const int r = 4 * (w0 + w) + b4;
            if (lane == 0 && r < r1)
              atomicAdd(&part[batch.base[ck] + r], (unsigned long long)((long long)hi * 65536 + (long long)lo));
          }
        }
      }
    }
  }
  __syncthreads();
  for (int s = threadIdx.x; s < batch.n_samples; s += SUM_THREADS)
    if (part[s]) atomicAdd(&tsum[s], part[s]);
}

// Cross-chain agreement of dataset blockIdx.y: per pair of chains a < b, max and sum over i < j of |pi_a - pi_b| with
// pi_c = count_c / rows_c.  Each CTA walks tiles blockIdx.x, +gridDim.x, ...; per round it stages E elements of the
// tile for all C chains in shared memory, and its threads take (pair, element group) slots.  Writes the CTA's partials
// to part_max / part_sum [k][cta][pair]; the host reduces them over the CTAs in CTA order.
constexpr int SUM_AG_SMEM = 4096;  // doubles of staged PSM values per round (C x E)
constexpr int SUM_AG_PPT = 8;      // pairs per thread: C <= 64 gives at most 2016 pairs
__global__ void __launch_bounds__(SUM_THREADS) k_summary_agree(const unsigned* counts, const double* rows, int C,
                                                               size_t chain_stride, size_t k_stride, long long n, int T,
                                                               int tiles, double* part_max, double* part_sum) {
  __shared__ double pis[SUM_AG_SMEM];
  __shared__ uint8_t pa[2016], pb[2016];
  const int P2 = C * (C - 1) / 2;
  const int S = P2 < SUM_THREADS ? P2 : SUM_THREADS, G = SUM_THREADS / S;
  const int E = SUM_AG_SMEM / C >= SUM_TE ? SUM_TE : SUM_AG_SMEM / C;  // a power of two when C is; else floor
  const int k = blockIdx.y;
  for (int p = threadIdx.x; p < P2; p += SUM_THREADS) {
    int a = 0, r = p;
    while (r >= C - 1 - a) { r -= C - 1 - a; ++a; }
    pa[p] = (uint8_t)a;
    pb[p] = (uint8_t)(a + 1 + r);
  }
  const bool active = threadIdx.x < S * G;
  const int slot = threadIdx.x % S, g = threadIdx.x / S;
  double mx[SUM_AG_PPT], sm[SUM_AG_PPT];
#pragma unroll
  for (int u = 0; u < SUM_AG_PPT; ++u) mx[u] = sm[u] = 0.0;
  for (int t = blockIdx.x; t < tiles; t += gridDim.x) {
    int ti, tj;
    sum_tile_of(t, T, ti, tj);
    const unsigned* base = counts + (size_t)k * k_stride + (size_t)t * SUM_TE;
    for (int e0 = 0; e0 < SUM_TE; e0 += E) {
      __syncthreads();
      for (int idx = threadIdx.x; idx < C * E; idx += SUM_THREADS) {
        const int c = idx / E, e = e0 + idx % E;
        const long long i = (long long)ti * SUM_TILE + e / SUM_TILE, j = (long long)tj * SUM_TILE + e % SUM_TILE;
        pis[idx] = (e < SUM_TE && i < j && j < n) ? (double)base[c * chain_stride + e] / rows[c] : 0.0;
      }
      __syncthreads();
      if (active) {
        for (int e = g; e < E; e += G) {
#pragma unroll
          for (int u = 0; u < SUM_AG_PPT; ++u) {
            const int p = slot + u * S;
            if (p < P2) {
              const double d = fabs(pis[pa[p] * E + e] - pis[pb[p] * E + e]);
              mx[u] = fmax(mx[u], d);
              sm[u] += d;
            }
          }
        }
      }
    }
  }
  __syncthreads();
  double* out_max = part_max + ((size_t)k * gridDim.x + blockIdx.x) * P2;
  double* out_sum = part_sum + ((size_t)k * gridDim.x + blockIdx.x) * P2;
  if (G == 1) {
#pragma unroll
    for (int u = 0; u < SUM_AG_PPT; ++u) {
      const int p = slot + u * S;
      if (p < P2) { out_max[p] = mx[u]; out_sum[p] = sm[u]; }
    }
    return;
  }
  // G > 1: one pair per thread (P2 = S); the G groups' partials are combined in group order
  if (active) { pis[g * S + slot] = mx[0]; pis[SUM_THREADS + g * S + slot] = sm[0]; }
  __syncthreads();
  if (threadIdx.x < S) {
    double m = 0.0, s = 0.0;
    for (int q = 0; q < G; ++q) { m = fmax(m, pis[q * S + threadIdx.x]); s += pis[SUM_THREADS + q * S + threadIdx.x]; }
    out_max[threadIdx.x] = m;
    out_sum[threadIdx.x] = s;
  }
}

}  // namespace summary
