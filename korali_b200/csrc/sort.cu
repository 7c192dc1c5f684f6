// sort.cu — K4: fitness ranking. Replaces sort_index (CMAES.cpp.base:940-950: std::sort of indices by
// vec[i1] > vec[i2]). Definition (also the oracle's): descending F(x), ASCENDING INDEX among equal values.
//
// Hand-written LSD radix sort (no CUB/Thrust): 64-bit order-preserving keys (descending), 8 passes of 8 bits,
// each pass = per-block digit histogram -> single-block exclusive scan -> stable scatter. Stability inside a
// block comes from warp-striped ownership + __match_any_sync ranks, so equal keys keep ascending index.
// The whole sorted order is produced (weights depend on the rank of every one of the top-mu samples).
#include <cooperative_groups.h>

#include "common.cuh"
#include "kernels.h"

namespace kc {

namespace {
constexpr int SORT_THREADS = 256;
constexpr int SORT_ITEMS = 8;
constexpr int SORT_TILE = SORT_THREADS * SORT_ITEMS;  // 2048 keys per block

__device__ __forceinline__ unsigned long long desc_key(double f) {
  if (f == 0.0) f = 0.0;  // -0.0 == +0.0 for the reference comparator
  unsigned long long u = (unsigned long long)__double_as_longlong(f);
  const unsigned long long asc = (u >> 63) ? ~u : (u | 0x8000000000000000ull);
  return ~asc;
}
}  // namespace

__global__ void __launch_bounds__(256) sort_make_keys_kernel(const double* __restrict__ f, int n, unsigned long long* __restrict__ keys,
                                                             unsigned* __restrict__ vals) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    keys[i] = desc_key(f[i]);
    vals[i] = (unsigned)i;
  }
}

__global__ void __launch_bounds__(SORT_THREADS) sort_hist_kernel(const unsigned long long* __restrict__ keys, int n, int shift,
                                                                 unsigned* __restrict__ hist, int nblocks) {
  __shared__ unsigned h[256];
  h[threadIdx.x] = 0;
  __syncthreads();
  const int base = blockIdx.x * SORT_TILE;
#pragma unroll
  for (int r = 0; r < SORT_ITEMS; r++) {
    const int i = base + r * SORT_THREADS + threadIdx.x;
    if (i < n) atomicAdd(&h[(unsigned)(keys[i] >> shift) & 255u], 1u);
  }
  __syncthreads();
  hist[threadIdx.x * nblocks + blockIdx.x] = h[threadIdx.x];
}

// Exclusive scan of hist[256 * nblocks] (digit-major) in place, single block of 1024 threads.
__global__ void __launch_bounds__(1024) sort_scan_kernel(unsigned* __restrict__ hist, int total) {
  __shared__ unsigned warp_tot[32];
  __shared__ unsigned carry;
  if (threadIdx.x == 0) carry = 0;
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int base = 0; base < total; base += 1024) {
    const int i = base + threadIdx.x;
    const unsigned v = i < total ? hist[i] : 0u;
    unsigned x = v;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
      const unsigned y = __shfl_up_sync(0xffffffffu, x, off);
      if (lane >= off) x += y;
    }
    if (lane == 31) warp_tot[warp] = x;
    __syncthreads();
    if (warp == 0) {
      unsigned w = warp_tot[lane];
#pragma unroll
      for (int off = 1; off < 32; off <<= 1) {
        const unsigned y = __shfl_up_sync(0xffffffffu, w, off);
        if (lane >= off) w += y;
      }
      warp_tot[lane] = w;  // inclusive over warps
    }
    __syncthreads();
    const unsigned warp_base = warp ? warp_tot[warp - 1] : 0u;
    const unsigned c = carry;
    if (i < total) hist[i] = c + warp_base + x - v;
    __syncthreads();
    if (threadIdx.x == 1023) carry = c + warp_base + x;
    __syncthreads();
  }
}

__global__ void __launch_bounds__(SORT_THREADS)
sort_scatter_kernel(const unsigned long long* __restrict__ keys_in, const unsigned* __restrict__ vals_in,
                    unsigned long long* __restrict__ keys_out, unsigned* __restrict__ vals_out, int n, int shift,
                    const unsigned* __restrict__ offsets, int nblocks) {
  __shared__ unsigned wcount[SORT_THREADS / 32][256];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int i = threadIdx.x; i < (SORT_THREADS / 32) * 256; i += SORT_THREADS) (&wcount[0][0])[i] = 0;
  __syncthreads();
  // warp-striped ownership: warp w owns keys [base + w*256, base + (w+1)*256), consumed 32 at a time in order
  const int base = blockIdx.x * SORT_TILE + warp * (32 * SORT_ITEMS);
  unsigned long long k[SORT_ITEMS];
  unsigned v[SORT_ITEMS], loc[SORT_ITEMS], dig[SORT_ITEMS];
  const unsigned lt = (1u << lane) - 1u;
#pragma unroll
  for (int r = 0; r < SORT_ITEMS; r++) {
    const int i = base + r * 32 + lane;
    const bool ok = i < n;
    k[r] = ok ? keys_in[i] : 0ull;
    v[r] = ok ? vals_in[i] : 0u;
    dig[r] = ok ? ((unsigned)(k[r] >> shift) & 255u) : 0xffffffffu;
    const unsigned peers = __match_any_sync(0xffffffffu, dig[r]);
    unsigned old = 0;
    if (ok) old = wcount[warp][dig[r]];
    __syncwarp();
    if (ok && (peers & lt) == 0) wcount[warp][dig[r]] = old + __popc(peers);  // group leader = lowest lane
    __syncwarp();
    loc[r] = old + __popc(peers & lt);
  }
  __syncthreads();
  {
    const int d = threadIdx.x;  // 256 threads <-> 256 digits
    unsigned running = offsets[d * nblocks + blockIdx.x];
#pragma unroll
    for (int w = 0; w < SORT_THREADS / 32; w++) {
      const unsigned c = wcount[w][d];
      wcount[w][d] = running;
      running += c;
    }
  }
  __syncthreads();
#pragma unroll
  for (int r = 0; r < SORT_ITEMS; r++) {
    if (dig[r] != 0xffffffffu) {
      const unsigned pos = wcount[warp][dig[r]] + loc[r];
      keys_out[pos] = k[r];
      vals_out[pos] = v[r];
    }
  }
}

// ---- the eight passes in ONE cooperative launch (populations up to one 2048-key tile per SM) -----------------------------------
// A pass keeps its tile in registers between the histogram and the scatter (the three-launch version reads it twice), the digit
// offsets of a CTA are formed by the CTA itself from the block-major histogram table (256 threads <-> 256 digits, 32 coalesced
// loads each at lambda = 65536), and the passes are separated by grid barriers instead of launch boundaries: 25 launches of a
// few microseconds each become one. Same warp-striped ownership and ranks as sort_scatter_kernel: the order is bit-identical.
__global__ void __launch_bounds__(SORT_THREADS)
sort_fused_kernel(const double* __restrict__ f, int n, unsigned long long* k0, unsigned long long* k1, unsigned* v0, unsigned* v1,
                  unsigned* sorted_idx, unsigned* hist) {   // (the ping-pong buffers change roles per pass: no __restrict__, L2 loads)
  namespace cg = cooperative_groups;
  cg::grid_group grid = cg::this_grid();
  __shared__ unsigned wcount[SORT_THREADS / 32][256];
  __shared__ unsigned wtot[SORT_THREADS / 32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nblocks = gridDim.x;
  const int base = blockIdx.x * SORT_TILE + warp * (32 * SORT_ITEMS);
  const unsigned lt = (1u << lane) - 1u;
  for (int pass = 0; pass < 8; pass++) {
    const int shift = 8 * pass;
    for (int i = threadIdx.x; i < (SORT_THREADS / 32) * 256; i += SORT_THREADS) (&wcount[0][0])[i] = 0;
    __syncthreads();
    unsigned long long k[SORT_ITEMS];
    unsigned v[SORT_ITEMS], loc[SORT_ITEMS], dig[SORT_ITEMS];
#pragma unroll
    for (int r = 0; r < SORT_ITEMS; r++) {
      const int i = base + r * 32 + lane;
      const bool ok = i < n;
      if (pass == 0) { k[r] = ok ? desc_key(f[i]) : 0ull; v[r] = (unsigned)i; }
      else { k[r] = ok ? __ldcg(k0 + i) : 0ull; v[r] = ok ? __ldcg(v0 + i) : 0u; }
      dig[r] = ok ? ((unsigned)(k[r] >> shift) & 255u) : 0xffffffffu;
      const unsigned peers = __match_any_sync(0xffffffffu, dig[r]);
      unsigned old = 0;
      if (ok) old = wcount[warp][dig[r]];
      __syncwarp();
      if (ok && (peers & lt) == 0) wcount[warp][dig[r]] = old + __popc(peers);
      __syncwarp();
      loc[r] = old + __popc(peers & lt);
    }
    __syncthreads();
    const int d = threadIdx.x;
    unsigned mine = 0;
#pragma unroll
    for (int w = 0; w < SORT_THREADS / 32; w++) mine += wcount[w][d];
    hist[blockIdx.x * 256 + d] = mine;
    __threadfence();
    grid.sync();
    // offset of digit d in this block = keys with a smaller digit anywhere + keys with digit d in earlier blocks
    unsigned total = 0, before = 0;
    for (int b = 0; b < nblocks; b++) {
      const unsigned c = __ldcg(hist + b * 256 + d);
      if (b < (int)blockIdx.x) before += c;
      total += c;
    }
    unsigned x = total;   // exclusive scan of the digit totals over the 256 threads
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) { const unsigned y = __shfl_up_sync(0xffffffffu, x, off); if (lane >= off) x += y; }
    if (lane == 31) wtot[warp] = x;
    __syncthreads();
    unsigned wbase = 0;
#pragma unroll
    for (int w = 0; w < SORT_THREADS / 32; w++) if (w < warp) wbase += wtot[w];
    unsigned running = wbase + x - total + before;
#pragma unroll
    for (int w = 0; w < SORT_THREADS / 32; w++) {
      const unsigned c = wcount[w][d];
      wcount[w][d] = running;
      running += c;
    }
    __syncthreads();
    unsigned* vout = (pass == 7) ? sorted_idx : v1;
#pragma unroll
    for (int r = 0; r < SORT_ITEMS; r++) {
      if (dig[r] != 0xffffffffu) {
        const unsigned pos = wcount[warp][dig[r]] + loc[r];
        if (pass < 7) k1[pos] = k[r];
        vout[pos] = v[r];
      }
    }
    __threadfence();
    grid.sync();
    unsigned long long* tk = k0; k0 = k1; k1 = tk;
    unsigned* tv = v0; v0 = v1; v1 = tv;
  }
}

// hist kernel uses block-striped reads; the scatter kernel uses warp-striped reads of the SAME tile, so the
// per-block histograms agree.
size_t sort_workspace_bytes(int n) {
  const int nblocks = (n + SORT_TILE - 1) / SORT_TILE;
  size_t b = 0;
  b += 2 * sizeof(unsigned long long) * (size_t)n;  // keys ping-pong
  b += 2 * sizeof(unsigned) * (size_t)n;            // vals ping-pong
  b += sizeof(unsigned) * 256 * (size_t)(nblocks > 0 ? nblocks : 1);
  return b + 1024;
}

// Sorts; the final order lands in sorted_idx (unsigned, length n). Returns number of kernel launches.
// ---- small populations: rank by counting (3 launches instead of 25) --------------------------------------------------
// rank_i = #{ j : key_j < key_i  or  (key_j == key_i and j < i) } on the same order-preserving descending keys, i.e. exactly
// the total order the stable radix passes produce (ascending index among equal values): bit-identical output. The n^2
// comparisons are spread over a 2-D grid (256 elements x 512 candidates per CTA, candidates staged in shared memory and
// read as broadcasts); partial counts meet in integer atomics, so the result does not depend on the execution order.
constexpr int RANK_MAX_N = 16384;
constexpr int RANK_CHUNK = 512;

__global__ void __launch_bounds__(256) sort_rank_count_kernel(const double* __restrict__ f, int n, unsigned* __restrict__ rank) {
  __shared__ unsigned long long sk[RANK_CHUNK];
  const int j0 = blockIdx.y * RANK_CHUNK;
  const int jn = min(RANK_CHUNK, n - j0);
  for (int j = threadIdx.x; j < jn; j += 256) sk[j] = desc_key(f[j0 + j]);
  __syncthreads();
  const int i = blockIdx.x * 256 + threadIdx.x;
  if (i >= n) return;
  const unsigned long long key = desc_key(f[i]);
  const int split = min(max(i - j0, 0), jn);   // candidates [0, split) have a smaller index than i: ties count
  unsigned r = 0;
  for (int j = 0; j < split; j++) r += sk[j] <= key ? 1u : 0u;
  for (int j = split; j < jn; j++) r += sk[j] < key ? 1u : 0u;
  if (r) atomicAdd(&rank[i], r);
}

__global__ void __launch_bounds__(256) sort_rank_scatter_kernel(const unsigned* __restrict__ rank, int n, unsigned* __restrict__ sorted_idx) {
  const int i = blockIdx.x * 256 + threadIdx.x;
  if (i < n) sorted_idx[rank[i]] = (unsigned)i;
}

int launch_sort_index(cudaStream_t st, const double* f, int n, void* workspace, unsigned* sorted_idx, int num_sms) {
  if (n <= 0) return 0;
  if (n <= RANK_MAX_N) {
    unsigned* rank = (unsigned*)workspace;
    cudaMemsetAsync(rank, 0, sizeof(unsigned) * (size_t)n, st);
    dim3 grid((n + 255) / 256, (n + RANK_CHUNK - 1) / RANK_CHUNK);
    sort_rank_count_kernel<<<grid, 256, 0, st>>>(f, n, rank);
    sort_rank_scatter_kernel<<<(n + 255) / 256, 256, 0, st>>>(rank, n, sorted_idx);
    return 2;
  }
  const int nblocks = (n + SORT_TILE - 1) / SORT_TILE;
  char* w = (char*)workspace;
  unsigned long long* k0 = (unsigned long long*)w; w += sizeof(unsigned long long) * (size_t)n;
  unsigned long long* k1 = (unsigned long long*)w; w += sizeof(unsigned long long) * (size_t)n;
  unsigned* v0 = (unsigned*)w; w += sizeof(unsigned) * (size_t)n;
  unsigned* v1 = (unsigned*)w; w += sizeof(unsigned) * (size_t)n;
  unsigned* hist = (unsigned*)w;
  if (nblocks <= num_sms) {   // one cooperative launch (every CTA must be resident: one tile per SM at most)
    const double* fp = f;
    void* args[] = {&fp, &n, &k0, &k1, &v0, &v1, &sorted_idx, &hist};
    if (cudaLaunchCooperativeKernel((const void*)sort_fused_kernel, dim3(nblocks), dim3(SORT_THREADS), args, 0, st) == cudaSuccess) return 1;
    cudaGetLastError();
  }
  int gk = (n + 255) / 256;
  if (gk > num_sms * 8) gk = num_sms * 8;
  sort_make_keys_kernel<<<gk, 256, 0, st>>>(f, n, k0, v0);
  int launches = 1;
  for (int pass = 0; pass < 8; pass++) {
    const int shift = 8 * pass;
    unsigned* vout = (pass == 7) ? sorted_idx : v1;
    sort_hist_kernel<<<nblocks, SORT_THREADS, 0, st>>>(k0, n, shift, hist, nblocks);
    sort_scan_kernel<<<1, 1024, 0, st>>>(hist, 256 * nblocks);
    sort_scatter_kernel<<<nblocks, SORT_THREADS, 0, st>>>(k0, v0, k1, vout, n, shift, hist, nblocks);
    launches += 3;
    unsigned long long* tk = k0; k0 = k1; k1 = tk;
    unsigned* tv = v0; v0 = v1; v1 = tv;
  }
  return launches;
}

}  // namespace kc
