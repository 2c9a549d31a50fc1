// meanshift.cu -- batched Gaussian mean-shift vote clustering for sm_100a.
//
// Replaces MeanShiftTorch.fit (reference pvn3d/lib/utils/meanshift_pytorch.py:13-51), which per
// iteration materialises four [n,n,3] float32 tensors with ~10 torch kernels and one host sync,
// and is called 1 + 1 + 8 times per object from a Python loop (pvn3d_eval_utils.py:53-57,84-97).
// Here ANY number of fits (every class of every frame, all keypoints) runs in four launches:
//
//   ms_setup     per-fit bookkeeping, tile prefix sums
//   ms_density   exact pass: num_in_i = #{j : |A_i - A_j| < bw}; arg-max with first-index ties
//                -> max_idx (meanshift_pytorch.py:46-49).  Distances use the fp32 contraction CPU
//                torch.norm uses (common.cuh: torch_sqnorm) and a pre-computed d^2 threshold that
//                is equivalent to `sqrtf(d2) < float(bw)`, so labels / counts are bit-exact.
//   ms_prepare   labels = |A[max_idx] - A_j| < bw (:50), origin = A[max_idx], centred copies
//   ms_iterate   ONE persistent cooperative kernel runs every iteration of every fit:
//                work items (fit, tile of seeds) are handed out by an atomic ticket, all seeds
//                of a tile sweep the fit's points from shared memory (broadcast LDS.128), and a
//                grid barrier per iteration applies the reference's GLOBAL stop rule per fit
//                (max_i |dC_i| < bw*1e-3 or it > max_iter, :39-42).  No host involvement.
//
// Arithmetic of the sweep: with points/seeds centred on A[max_idx] (a', c') and
// k = -log2(e)/(2 bw^2):  w_ij = 2^( k|a'|^2 + k|c'|^2 - 2k a'.c' )  -- 1 FADD + 3 FFMA + 1 MUFU.EX2
// per pair, then 1 FADD + 3 FFMA to accumulate sum(w), sum(w a').  The reference's constant
// 1/(bw sqrt(2 pi)) cancels in sum(w a)/sum(w) (SURVEY App. A.4.1 (iii)).  Centres agree with the
// CPU reference to ~1e-6 relative (tests pin 1e-4, BASELINE.json north_star); labels, counts and
// max_idx are exact.
#include <cooperative_groups.h>

#include <algorithm>
#include <cmath>

#include "common.cuh"

namespace cg = cooperative_groups;

namespace pvn3d {
namespace {

constexpr int kMsThreads = 256;
constexpr int kMsFitMax = 2048;  // fits per launch chunk (prefix array lives in shared memory)
constexpr int kMsPtTile = 4096;  // points per shared-memory tile of the sweep (64 KB)
constexpr int kMsPairs = kMsPtTile / 2;
constexpr int kMsDensTile = 1024;  // points per tile of the density pass (16 KB static)
constexpr int kMsWarps = kMsThreads / 32;
constexpr int kMsCfgInts = 4096;   // [0..2] phase tickets, [3] grid barrier, [4..2047] debug, [2048..] CTAs seen per SM
constexpr int kMsCfgSm = 2048;
constexpr int kMsPruneMax = 4096;   // points per fit the pruned density kernel keeps in shared memory
constexpr int kMsPruneBins = 2048;  // radial bins of its counting sort
constexpr int kMsCfgCertified = 8;  // statistics of the last launch: fits closed by ms_witness_kernel

struct MsArgs {
  const float4 *pts;
  const int *fit_start;
  const int *fit_count;
  int n_fits;
  float t2;           // d2 < t2  <=>  sqrtf(d2) < float(bandwidth)
  float stop_thresh;  // float(bandwidth * 1e-3)
  float eps_stat;     // early-exit stationarity threshold for the returned seed
  float kexp;         // -log2(e) / (2 bw^2)
  int max_iter;
  unsigned flags;
  // outputs
  float4 *ctr;
  uint8_t *labels;
  int *max_idx;
  int *n_in;
  // workspace
  float4 *cpts;
  float4 *seeds;
  unsigned long long *best_key;
  int *done;
  int *iters;        // T per fit
  int *star_it;      // first iteration at which the returned seed was stationary (0 = not yet)
  int *act;          // [3][cap]   work lists: indices (within the fit) of the seeds still moving
  int *act_cnt;      // [3][n_fits]
  unsigned *viol;    // [n_fits][viol_words] bit `it` = some seed moved >= stop_thresh at iteration it
  float4 *traj;      // [n_fits][traj_stride] positions of the returned seed per iteration
  int *dens_prefix;  // [n_fits+1]
  int *dens_cnt;     // [cap] inlier count of every input point (exact pass); witness selection
  float delta_path;  // certified mode: the returned seed's remaining path at it0 is below this
  int dens_pruned;   // fits of <= kMsPruneMax points are counted by ms_density_pruned_kernel
  float bwf;         // float(bandwidth)
  int *cfg;          // [0..2] ticket counters of the phases
  int cap;
  int viol_words;
  int traj_stride;
  int ctas_per_sm;   // co-resident CTAs of ms_iterate_kernel per SM (grid = ctas_per_sm * #SM)
};

__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// exclusive scan of one int per thread across the CTA; returns the exclusive prefix, *total = sum
template <int NT>
__device__ __forceinline__ int block_exclusive_scan(int v, int *s_warp /*[NT/32]*/, int *total) {
  const unsigned lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
  int incl = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int u = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += u;
  }
  if (lane == 31) s_warp[warp] = incl;
  __syncthreads();
  int wsum = (lane < NT / 32) ? s_warp[lane] : 0;
  int wincl = wsum;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int u = __shfl_up_sync(0xffffffffu, wincl, o);
    if (lane >= o) wincl += u;
  }
  const int wexcl = __shfl_sync(0xffffffffu, wincl - wsum, warp);
  *total = __shfl_sync(0xffffffffu, wincl, NT / 32 - 1);
  __syncthreads();  // s_warp reusable
  return wexcl + incl - v;
}

// largest f in [0, n) with prefix[f] <= x   (prefix non-decreasing, prefix[0] = 0 <= x)
__device__ __forceinline__ int find_segment(const int *prefix, int n, int x) {
  int lo = 0, hi = n - 1;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (prefix[mid] <= x) lo = mid; else hi = mid - 1;
  }
  return lo;
}

// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(1024) ms_setup_kernel(MsArgs a) {
  __shared__ int s_warp[32];
  __shared__ int s_run;
  const int t = threadIdx.x;
  if (t == 0) s_run = 0;
  __syncthreads();
  for (int f0 = 0; f0 < a.n_fits; f0 += 1024) {
    const int f = f0 + t;
    int cnt = 0;
    if (f < a.n_fits) {
      cnt = max(a.fit_count[f], 0);
      a.best_key[f] = 0ull;
      a.done[f] = cnt == 0;
      a.iters[f] = 0;
      a.star_it[f] = 0;
      a.act_cnt[f] = a.act_cnt[a.n_fits + f] = a.act_cnt[2 * a.n_fits + f] = 0;
      for (int w = 0; w < a.viol_words; ++w) a.viol[static_cast<size_t>(f) * a.viol_words + w] = 0u;
      if (cnt == 0) {
        a.ctr[f] = make_float4(0.f, 0.f, 0.f, 0.f);
        a.max_idx[f] = 0;
        a.n_in[f] = 0;
      }
    }
    int total;
    const int excl = block_exclusive_scan<1024>((cnt + kMsThreads - 1) / kMsThreads, s_warp, &total);
    const int run = s_run;
    if (f < a.n_fits) a.dens_prefix[f] = run + excl;
    __syncthreads();
    if (t == 0) s_run = run + total;
    __syncthreads();
  }
  if (t == 0) a.dens_prefix[a.n_fits] = s_run;
  for (int i = t; i < kMsCfgInts; i += 1024) a.cfg[i] = 0;
}

// ------------------------------------------------------------------------------------------------
// exact density pass: one thread per input point, all points of the fit swept from shared memory.
// The tile holds point PAIRS (x0,x1,y0,y1 | z0,z1) so that the distance of one seed to two points is
// three FADD2 + FMUL2 + two FFMA2 on the packed fp32 pipe: per lane these are the same IEEE operations in
// the same order as torch_sqnorm (fma(dz,dz, fma(dy,dy, dx*dx)) on p - me), so counts stay bit-exact, at
// 6 instead of 9 issue slots per pair test.
__global__ void __launch_bounds__(kMsThreads) ms_density_kernel(MsArgs a) {
  __shared__ float4 s_xy[kMsDensTile / 2];   // (x0, x1, y0, y1)
  __shared__ float2 s_z[kMsDensTile / 2];    // (z0, z1)
  __shared__ unsigned long long s_key[kMsWarps];
  const int tile = blockIdx.x;
  if (tile >= a.dens_prefix[a.n_fits]) return;
  const int f = find_segment(a.dens_prefix, a.n_fits, tile);
  const int start = a.fit_start[f], cnt = a.fit_count[f];
  if (a.dens_pruned && cnt <= kMsPruneMax) return;   // ms_density_pruned_kernel counts this fit
  const int i = (tile - a.dens_prefix[f]) * kMsThreads + threadIdx.x;
  const bool live = i < cnt;
  const float4 me = a.pts[start + (live ? i : 0)];
  const float2 nx = make_float2(-me.x, -me.x), ny = make_float2(-me.y, -me.y), nz = make_float2(-me.z, -me.z);
  const float t2 = a.t2;
  const float inf = __int_as_float(0x7f800000);
  int count = 0;
  for (int base = 0; base < cnt; base += kMsDensTile) {
    const int n = min(kMsDensTile, cnt - base);
    const int npairs = (n + 1) >> 1;
    __syncthreads();
    for (int q = threadIdx.x; q < npairs; q += kMsThreads) {
      const float4 p0 = a.pts[start + base + 2 * q];
      // odd tail: a point at infinity is never an inlier (inf < t2 is false)
      const float4 p1 = 2 * q + 1 < n ? a.pts[start + base + 2 * q + 1] : make_float4(inf, inf, inf, 0.f);
      s_xy[q] = make_float4(p0.x, p1.x, p0.y, p1.y);
      s_z[q] = make_float2(p0.z, p1.z);
    }
    __syncthreads();
#pragma unroll 4
    for (int j = 0; j < npairs; ++j) {
      const float4 xy = s_xy[j];
      const float2 z = s_z[j];
      // dis = torch.norm(Ar - Cr): diff = A_j - A_i   (meanshift_pytorch.py:46-48)
      const float2 dx = __fadd2_rn(make_float2(xy.x, xy.y), nx);
      const float2 dy = __fadd2_rn(make_float2(xy.z, xy.w), ny);
      const float2 dz = __fadd2_rn(z, nz);
      const float2 d2 = __ffma2_rn(dz, dz, __ffma2_rn(dy, dy, __fmul2_rn(dx, dx)));
      count += (d2.x < t2 ? 1 : 0) + (d2.y < t2 ? 1 : 0);
    }
  }
  if (live) a.dens_cnt[start + i] = count;
  unsigned long long key =
      live ? ((static_cast<unsigned long long>(count) << 32) | (0xFFFFFFFFu - static_cast<unsigned>(i)))
           : 0ull;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const unsigned long long other = __shfl_xor_sync(0xffffffffu, key, o);
    key = other > key ? other : key;
  }
  if ((threadIdx.x & 31) == 0) s_key[threadIdx.x >> 5] = key;
  __syncthreads();
  if (threadIdx.x == 0) {
#pragma unroll
    for (int w = 1; w < kMsWarps; ++w) key = s_key[w] > key ? s_key[w] : key;
    atomicMax(a.best_key + f, key);  // (count desc, index asc): torch.max first-index rule (:49)
  }
}

// ------------------------------------------------------------------------------------------------
// Exact density pass WITHOUT n^2 tests: num_in_i = #{j : |A_i - A_j| < bw} (meanshift_pytorch.py:46-48).
//
// Votes are a tight cluster plus scattered outliers.  With r_i = |A_i - c| for a pivot c near the cluster, the
// triangle inequality decides most pairs without looking at them:
//     r_i + r_j < bw - eps    =>  |A_i - A_j| < bw      (certainly an inlier of i)
//     |r_i - r_j| > bw + eps  =>  |A_i - A_j| > bw      (certainly not)
// One CTA per fit sorts its points by r (counting sort over radial bins, all in shared memory); point i then
// needs   count_i = #{j : r_j < bw - eps - r_i}   -- a prefix sum, no distance evaluated --   plus an exact test
// (the same fp32 contraction and threshold as the brute-force pass) of the points whose r_j lies in the band
// [max(bw - eps - r_i, r_i - bw - eps), r_i + bw + eps].  For an inlier (r_i ~ 1 cm, bw = 8 cm) the band holds the
// few outliers 7-9 cm from the pivot; for an outlier it is a thin shell of other outliers.  eps (0.1 mm + 1e-5 of
// the cloud's radius) dwarfs every fp32 rounding involved, so each pair gets exactly the verdict the brute-force
// test would give: counts, arg-max and labels stay bit-exact (tests: all golden cases + a direct comparison
// against the brute-force kernel).  The pivot only steers how much is pruned, never the result: three rounds of
// "mean of the points near the current estimate" starting from the centroid.
struct MsPruneSmem {
  float4 pts[kMsPruneMax];        // original order: x, y, z, r
  int idx_sorted[kMsPruneMax];    // point indices in order of increasing radius
  int cursor[kMsPruneBins + 1];   // scatter cursors of the counting sort (+ overflow bin)
  int bin_start[kMsPruneBins + 2];   // [kMsPruneBins] = first point of the overflow bin (non-finite coordinates)
  float red[kMsWarps][4];
  float4 pivot;
  float max_r;
  unsigned long long key[kMsWarps];
};

__device__ __forceinline__ float4 ms_block_sum4(MsPruneSmem &sm, float4 v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    v.x += __shfl_xor_sync(0xffffffffu, v.x, o);
    v.y += __shfl_xor_sync(0xffffffffu, v.y, o);
    v.z += __shfl_xor_sync(0xffffffffu, v.z, o);
    v.w += __shfl_xor_sync(0xffffffffu, v.w, o);
  }
  __syncthreads();
  if ((threadIdx.x & 31) == 0) {
    sm.red[threadIdx.x >> 5][0] = v.x; sm.red[threadIdx.x >> 5][1] = v.y;
    sm.red[threadIdx.x >> 5][2] = v.z; sm.red[threadIdx.x >> 5][3] = v.w;
  }
  __syncthreads();
  float4 t = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
  for (int w = 0; w < kMsWarps; ++w) {
    t.x += sm.red[w][0]; t.y += sm.red[w][1]; t.z += sm.red[w][2]; t.w += sm.red[w][3];
  }
  return t;   // identical in every thread
}

__global__ void __launch_bounds__(kMsThreads, 2) ms_density_pruned_kernel(MsArgs a) {
  extern __shared__ __align__(16) unsigned char ms_smem_raw[];
  MsPruneSmem &sm = *reinterpret_cast<MsPruneSmem *>(ms_smem_raw);
  const int f = blockIdx.x;
  const int n = a.fit_count[f];
  if (n <= 0 || n > kMsPruneMax) return;
  const int start = a.fit_start[f];
  const int t = threadIdx.x;
  const float bw = a.bwf, t2 = a.t2;

  // ---- points into shared memory, pivot = robust centre ------------------------------------------------
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  // (points with a NaN / inf coordinate never count and are never counted in the brute-force pass -- every
  // distance to them is NaN or inf; here they are kept out of the pivot and parked in an overflow bin)
  for (int i = t; i < n; i += kMsThreads) {
    const float4 p = a.pts[start + i];
    sm.pts[i] = make_float4(p.x, p.y, p.z, 0.f);
    if (fabsf(p.x) + fabsf(p.y) + fabsf(p.z) < __int_as_float(0x7f800000)) { acc.x += p.x; acc.y += p.y; acc.z += p.z; acc.w += 1.f; }
  }
  float4 sum = ms_block_sum4(sm, acc);
  float3 c = sum.w > 0.f ? make_float3(sum.x / sum.w, sum.y / sum.w, sum.z / sum.w) : make_float3(0.f, 0.f, 0.f);
#pragma unroll 1
  for (int round = 0; round < 2; ++round) {
    const float rad = round == 0 ? 2.f * bw : bw;
    acc = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int i = t; i < n; i += kMsThreads) {
      const float4 p = sm.pts[i];
      const float dx = p.x - c.x, dy = p.y - c.y, dz = p.z - c.z;
      if (dx * dx + dy * dy + dz * dz < rad * rad) { acc.x += p.x; acc.y += p.y; acc.z += p.z; acc.w += 1.f; }   // false for NaN
    }
    sum = ms_block_sum4(sm, acc);
    if (sum.w > 0.f) c = make_float3(sum.x / sum.w, sum.y / sum.w, sum.z / sum.w);
  }

  // ---- radii, bins, counting sort by radius ---------------------------------------------------------------
  float rmax = 0.f;
  for (int i = t; i < n; i += kMsThreads) {
    float4 p = sm.pts[i];
    const float dx = p.x - c.x, dy = p.y - c.y, dz = p.z - c.z;
    p.w = sqrtf(dx * dx + dy * dy + dz * dz);
    sm.pts[i] = p;
    if (p.w < __int_as_float(0x7f800000)) rmax = fmaxf(rmax, p.w);   // finite radii only
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) rmax = fmaxf(rmax, __shfl_xor_sync(0xffffffffu, rmax, o));
  __syncthreads();
  if ((t & 31) == 0) sm.red[t >> 5][0] = rmax;
  for (int b = t; b <= kMsPruneBins + 1; b += kMsThreads) sm.bin_start[b] = 0;
  __syncthreads();
  rmax = sm.red[0][0];
#pragma unroll
  for (int w = 1; w < kMsWarps; ++w) rmax = fmaxf(rmax, sm.red[w][0]);
  const float eps = 1e-4f + 1e-5f * (rmax + fabsf(c.x) + fabsf(c.y) + fabsf(c.z));
  const float inv_w = static_cast<float>(kMsPruneBins) / (rmax * 1.0001f + 1e-20f);
  auto bin_of = [&](float r) {
    const float x = r * inv_w;   // may be huge when every point coincides (rmax = 0): clamp before the conversion
    return x >= static_cast<float>(kMsPruneBins - 1) ? kMsPruneBins - 1 : max(0, static_cast<int>(x));
  };
  auto bin_of_point = [&](float r) { return r < __int_as_float(0x7f800000) ? bin_of(r) : kMsPruneBins; };   // overflow bin
  for (int i = t; i < n; i += kMsThreads) atomicAdd(&sm.bin_start[bin_of_point(sm.pts[i].w) + 1], 1);   // histogram, shifted by one
  __syncthreads();
  {  // inclusive scan of the shifted histogram = exclusive bin starts; 8 bins per thread
    constexpr int per = kMsPruneBins / kMsThreads;
    int local[per];
    int s_ = 0;
#pragma unroll
    for (int q = 0; q < per; ++q) { s_ += sm.bin_start[1 + t * per + q]; local[q] = s_; }
    int incl = s_;
    const unsigned lane = t & 31u;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int u = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += u;
    }
    __shared__ int s_warp[kMsWarps];
    if (lane == 31) s_warp[t >> 5] = incl;
    __syncthreads();
    int base = incl - s_;
    for (int w = 0; w < (t >> 5); ++w) base += s_warp[w];
#pragma unroll
    for (int q = 0; q < per; ++q) sm.bin_start[1 + t * per + q] = base + local[q];
  }
  __syncthreads();
  if (t == 0) sm.bin_start[kMsPruneBins + 1] += sm.bin_start[kMsPruneBins];   // overflow bin: [n_finite, n)
  __syncthreads();
  const int n_fin = sm.bin_start[kMsPruneBins];   // finite points come first in the sorted order
  // scatter: cursor per bin = its start (kept in r_sorted's storage as ints until the points land)
  int *cursor = sm.cursor;
  for (int b = t; b <= kMsPruneBins; b += kMsThreads) cursor[b] = sm.bin_start[b];
  __syncthreads();
  for (int i = t; i < n; i += kMsThreads) {
    const int pos = atomicAdd(&cursor[bin_of_point(sm.pts[i].w)], 1);
    sm.idx_sorted[pos] = i;
  }
  __syncthreads();

  // ---- counts ---------------------------------------------------------------------------------------------
  const float bw_lo = bw - eps, bw_hi = bw + eps;
  unsigned long long best = 0ull;
  for (int q = t; q < n; q += kMsThreads) {   // consecutive threads = consecutive radii: similar bands inside a warp
    const int i = sm.idx_sorted[q];
    const float4 me = sm.pts[i];
    const float lo = bw_lo - me.w, hi = me.w + bw_hi;
    int count = 0, first = 0;
    if (q >= n_fin) {
      first = n_fin;                           // non-finite point: empty band, count 0 (as every test on it fails)
    } else if (lo > 0.f) {
      first = sm.bin_start[bin_of(lo)];       // every point of an earlier bin has r_j < lo: certainly within bw of i
      count = first;
    } else {
      first = sm.bin_start[bin_of(fmaxf(me.w - bw_hi, 0.f))];   // earlier bins: r_j < r_i - bw - eps, certainly outside
    }
    const int last = q >= n_fin ? n_fin : (hi * inv_w >= static_cast<float>(kMsPruneBins) ? n_fin : sm.bin_start[bin_of(hi) + 1]);
    for (int pos = first; pos < last; ++pos) {
      const float4 p = sm.pts[sm.idx_sorted[pos]];
      // dis = torch.norm(Ar - Cr): diff = A_j - A_i, exactly as the brute-force pass
      count += torch_sqnorm(p.x - me.x, p.y - me.y, p.z - me.z) < t2 ? 1 : 0;
    }
    a.dens_cnt[start + i] = count;
    const unsigned long long key = (static_cast<unsigned long long>(count) << 32) | (0xFFFFFFFFu - static_cast<unsigned>(i));
    best = key > best ? key : best;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const unsigned long long other = __shfl_xor_sync(0xffffffffu, best, o);
    best = other > best ? other : best;
  }
  if ((t & 31) == 0) sm.key[t >> 5] = best;
  __syncthreads();
  if (t == 0) {
#pragma unroll
    for (int w = 1; w < kMsWarps; ++w) best = sm.key[w] > best ? sm.key[w] : best;
    a.best_key[f] = best;   // (count desc, index asc): torch.max first-index rule (:49); the only writer for this fit
  }
}

// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kMsThreads) ms_prepare_kernel(MsArgs a) {
  const int tile = blockIdx.x;
  if (tile >= a.dens_prefix[a.n_fits]) return;
  const int f = find_segment(a.dens_prefix, a.n_fits, tile);
  const int start = a.fit_start[f], cnt = a.fit_count[f];
  const int i = (tile - a.dens_prefix[f]) * kMsThreads + threadIdx.x;
  const unsigned long long key = a.best_key[f];
  const int mi = static_cast<int>(0xFFFFFFFFu - static_cast<unsigned>(key & 0xFFFFFFFFull));
  if (i == 0) {
    a.max_idx[f] = mi;
    a.n_in[f] = static_cast<int>(key >> 32);
    a.act_cnt[f] = cnt;  // phase 0 works on every seed
  }
  if (i >= cnt) return;
  a.act[start + i] = i;
  const float4 o = a.pts[start + mi];
  const float4 p = a.pts[start + i];
  const float dx = p.x - o.x, dy = p.y - o.y, dz = p.z - o.z;
  if (a.labels) a.labels[start + i] = torch_sqnorm(dx, dy, dz) < a.t2 ? 1 : 0;  // (:50)
  a.cpts[start + i] = make_float4(dx, dy, dz, a.kexp * (dx * dx + dy * dy + dz * dz));
  a.seeds[start + i] = make_float4(dx, dy, dz, 0.f);  // C <- A.clone()  (:31)
}

// ------------------------------------------------------------------------------------------------
// The iterations.
//
// Every seed's trajectory depends only on its own position and the (fixed) points, so seeds need
// not advance in lock step.  The reference's GLOBAL stop rule -- stop at the first iteration T whose
// largest shift over ALL seeds is below bw*1e-3 -- is recovered from a per-fit bitmask:
//   viol[f] bit `it` is set by any seed whose shift at iteration `it` is >= the threshold;
//   T = the first iteration whose bit is clear (or max_iter+1).
// A seed whose shift drops below eps = bw*1e-6 (1000x under the threshold) is FROZEN: it can no
// longer set a bit (its shift cannot grow 1000x again without moving ~9 cm, DESIGN.md section 5) and
// moves by < 1e-7 m from then on, so it is dropped from the work list.  The returned seed ("star",
// the densest input point) logs its position at every iteration, so C[max_idx] AFTER EXACTLY T
// iterations is what comes back, as in the reference.
//
// Work is organised in PHASES of several iterations (6,10,16,16,...): a tile of seeds keeps
// its seeds in registers and -- when the fit has <= 4096 points -- the whole point set in shared
// memory for the entire phase; between phases the still-moving seeds are compacted into dense
// tiles and a grid barrier lets every CTA take the same per-fit decisions.  Typical vote sets
// (tight cluster + 10 % outliers) need ~140 iterations by the reference's rule, but after the
// first phase only the few creeping outlier seeds are still in the lists.
// ------------------------------------------------------------------------------------------------
// Grid-wide barrier for the persistent kernel (all CTAs co-resident: cooperative launch).  The
// cooperative-groups grid.sync() spins on an acquire load, for which ptxas emits CCTL.IVALL (L1
// invalidate) in the polling loop: CTAs that ran out of tiles then hammer the L1/shared-memory pipe
// of their SM and slow the CTAs still sweeping by an order of magnitude (measured: 30 us per
// iteration instead of ~1 us in the late phases).  Here idle CTAs poll a monotonically increasing
// counter with relaxed loads and sleep in between; one fence pair orders the data.
__device__ __forceinline__ void ms_grid_barrier(unsigned *counter, unsigned &epoch) {
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();  // release: this CTA's global writes of the phase
    const unsigned target = (epoch + 1u) * gridDim.x;
    atomicAdd(counter, 1u);
    unsigned seen;
    for (;;) {
      asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(seen) : "l"(counter) : "memory");
      if (seen >= target) break;
      __nanosleep(256);
    }
    __threadfence();  // acquire: other CTAs' writes are visible from here on
  }
  ++epoch;
  __syncthreads();
}

struct MsIterSmem {
  float4 pts[kMsPtTile];
  int prefix[kMsFitMax + 1];
  int warp_scan[kMsWarps];
  int ticket;
};

__device__ __forceinline__ int ms_phase_end(int p) {  // last iteration of phase p
  // 1, 2, 3, 4, 6, 8, 12, 16, 32, 48, ...: T is detected at phase ends, so short phases bound the work
  // done past T; and the seeds that froze leave the work lists at phase ends -- most seeds of a vote
  // cluster are stationary after ~4 iterations, an order of magnitude fewer stay for the long tail
  if (p < 4) return p + 1;
  if (p < 6) return 6 + 2 * (p - 4);
  return p == 6 ? 12 : 16 * (p - 6);
}

// Shared-memory layout of a fit's points: point PAIRS, structure-of-arrays inside the pair
//   s_pts[p] = (x0, x1, y0, y1)      s_pts[kMsPairs + p] = (z0, z1, w0, w1)       w = k |a'|^2
// (two planes, so that a warp whose lanes read CONSECUTIVE pairs touches every bank once)
// so that the sweep runs on the packed FP32 pipe (FFMA2 / FADD2: two points per instruction):
// per point pair and seed 4 packed ops for the exponents, 2 MUFU.EX2, 4 packed ops to accumulate --
// 5 issue slots per pair evaluation instead of 9.  An odd tail is padded with w = -inf (weight 0).
__device__ __forceinline__ void ms_stage_pairs(float4 *s_pts, const float4 *__restrict__ cpts, int n) {
  const int npairs = (n + 1) >> 1;
  for (int q = threadIdx.x; q < npairs; q += kMsThreads) {
    const float4 p0 = cpts[2 * q];
    float4 p1 = make_float4(0.f, 0.f, 0.f, -__int_as_float(0x7f800000));
    if (2 * q + 1 < n) p1 = cpts[2 * q + 1];
    s_pts[q] = make_float4(p0.x, p1.x, p0.y, p1.y);
    s_pts[kMsPairs + q] = make_float4(p0.z, p1.z, p0.w, p1.w);
  }
}

struct MsSeedQ {  // per-seed constants of the exponent, duplicated into both halves of a pair
  float2 qx, qy, qz, qw;
};
struct MsSeedS {  // packed partial sums (even points, odd points)
  float2 sw, sx, sy, sz;
};
__device__ __forceinline__ MsSeedQ ms_seed_q(float k, float cx, float cy, float cz) {
  MsSeedQ q;
  const float x = -2.f * k * cx, y = -2.f * k * cy, z = -2.f * k * cz;
  const float w = k * (cx * cx + cy * cy + cz * cz);
  q.qx = make_float2(x, x); q.qy = make_float2(y, y); q.qz = make_float2(z, z); q.qw = make_float2(w, w);
  return q;
}
__device__ __forceinline__ void ms_pair_step(const float4 &A, const float4 &B, const MsSeedQ &q, MsSeedS &s) {
  const float2 x2 = make_float2(A.x, A.y), y2 = make_float2(A.z, A.w), z2 = make_float2(B.x, B.y),
               w2 = make_float2(B.z, B.w);
  const float2 e = __ffma2_rn(x2, q.qx, __ffma2_rn(y2, q.qy, __ffma2_rn(z2, q.qz, __fadd2_rn(w2, q.qw))));
  const float2 w = make_float2(ex2_approx(e.x), ex2_approx(e.y));
  s.sw = __fadd2_rn(s.sw, w);
  s.sx = __ffma2_rn(w, x2, s.sx);
  s.sy = __ffma2_rn(w, y2, s.sy);
  s.sz = __ffma2_rn(w, z2, s.sz);
}

template <int R>
__device__ __forceinline__ void ms_sweep(const float4 *__restrict__ s_pts, int npairs, const MsSeedQ (&q)[R],
                                         MsSeedS (&s)[R]) {
#pragma unroll 2
  for (int p = 0; p < npairs; ++p) {
    const float4 A = s_pts[p], B = s_pts[kMsPairs + p];  // broadcast LDS.128 x2
#pragma unroll
    for (int r = 0; r < R; ++r) ms_pair_step(A, B, q[r], s[r]);
  }
}

template <int R>
__device__ __forceinline__ void ms_run_tile(const MsArgs &a, MsIterSmem &sm, int f, int tile,
                                            int it_lo, int it_hi, int cur, int nxt) {
  const int start = a.fit_start[f], n_c = a.fit_count[f];
  const int n_act = a.act_cnt[static_cast<size_t>(cur) * a.n_fits + f];
  const int *act_cur = a.act + static_cast<size_t>(cur) * a.cap + start;
  int *act_nxt = a.act + static_cast<size_t>(nxt) * a.cap + start;
  const int t = threadIdx.x;
  const unsigned lane = t & 31u;
  const float k = a.kexp;
  const bool single = n_c <= kMsPtTile;  // whole point set stays in shared memory for the phase
  const bool freeze_on = !(a.flags & PVN3D_MS_NO_FREEZE);
  const int star = a.max_idx[f];

  int idx[R];
  float cx[R], cy[R], cz[R], last[R];
  bool frozen[R];
#pragma unroll
  for (int r = 0; r < R; ++r) {
    const int pos = tile * (kMsThreads * R) + r * kMsThreads + t;
    const bool valid = pos < n_act;
    idx[r] = valid ? act_cur[pos] : -1;
    const float4 c = a.seeds[start + (valid ? idx[r] : 0)];
    cx[r] = c.x; cy[r] = c.y; cz[r] = c.z; last[r] = c.w;
    frozen[r] = !valid;
  }
  __syncthreads();  // previous tile's readers are done with sm.pts
  if (single) {
    ms_stage_pairs(sm.pts, a.cpts + start, n_c);
    __syncthreads();
  }

  for (int it = it_lo; it <= it_hi; ++it) {
    bool live = false;
#pragma unroll
    for (int r = 0; r < R; ++r) live |= !frozen[r];
    const bool warp_live = __any_sync(0xffffffffu, live);
    if (single && !warp_live) break;  // no barriers inside the loop in single-tile mode

    MsSeedQ sq[R];
    MsSeedS ss[R];
#pragma unroll
    for (int r = 0; r < R; ++r) {
      sq[r] = ms_seed_q(k, cx[r], cy[r], cz[r]);
      ss[r].sw = ss[r].sx = ss[r].sy = ss[r].sz = make_float2(0.f, 0.f);
    }
    if (single) {
      ms_sweep<R>(sm.pts, (n_c + 1) >> 1, sq, ss);
    } else {
      for (int base = 0; base < n_c; base += kMsPtTile) {
        const int n = min(kMsPtTile, n_c - base);
        __syncthreads();
        ms_stage_pairs(sm.pts, a.cpts + start + base, n);
        __syncthreads();
        if (warp_live) ms_sweep<R>(sm.pts, (n + 1) >> 1, sq, ss);
      }
    }
    bool violates = false;
#pragma unroll
    for (int r = 0; r < R; ++r) {
      if (!frozen[r]) {
        // new_C = sum(w*A)/sum(w); Adis = |new_C - C|   (meanshift_pytorch.py:37-39)
        const float swr = ss[r].sw.x + ss[r].sw.y;
        const float nx = __fdiv_rn(ss[r].sx.x + ss[r].sx.y, swr), ny = __fdiv_rn(ss[r].sy.x + ss[r].sy.y, swr),
                    nz = __fdiv_rn(ss[r].sz.x + ss[r].sz.y, swr);
        const float sh = __fsqrt_rn(torch_sqnorm(nx - cx[r], ny - cy[r], nz - cz[r]));
        cx[r] = nx; cy[r] = ny; cz[r] = nz; last[r] = sh;
        violates |= !(sh < a.stop_thresh);
        const bool still = sh < a.eps_stat;
        if (idx[r] == star) {
          a.traj[static_cast<size_t>(f) * a.traj_stride + it] = make_float4(nx, ny, nz, sh);
          if (still && a.star_it[f] == 0) a.star_it[f] = it;  // only this thread ever writes it
        }
        if (still && freeze_on) frozen[r] = true;
      }
    }
    if (__any_sync(0xffffffffu, violates) && lane == 0)
      atomicOr(a.viol + static_cast<size_t>(f) * a.viol_words + (it >> 5), 1u << (it & 31));
    if (!single) {
      bool live2 = false;
#pragma unroll
      for (int r = 0; r < R; ++r) live2 |= !frozen[r];
      if (!__syncthreads_or(live2 ? 1 : 0)) break;
    }
  }

  // write the seeds back; the ones still moving go to the next phase's list
#pragma unroll
  for (int r = 0; r < R; ++r) {
    const bool valid = idx[r] >= 0;
    if (valid) a.seeds[start + idx[r]] = make_float4(cx[r], cy[r], cz[r], last[r]);
    const bool keep = valid && !frozen[r];
    const unsigned m = __ballot_sync(0xffffffffu, keep);
    if (m) {
      int base = 0;
      if (lane == 0) base = atomicAdd(a.act_cnt + static_cast<size_t>(nxt) * a.n_fits + f, __popc(m));
      base = __shfl_sync(0xffffffffu, base, 0);
      if (keep) act_nxt[base + __popc(m & lanemask_lt())] = idx[r];
    }
  }
}

// Split-sweep variant for the late phases, when only a few (creeping) seeds per fit are left: a
// seed's iterations are inherently sequential, so with one thread per seed the critical path is
// T * n_c pair evaluations of ONE lane.  Here a warp owns two seeds at a time and its 32 lanes share
// the sweep (lane l takes points l, l+32, ...); the eight partial sums are combined with a butterfly
// of warp shuffles, so every lane holds the same totals and the same new position.  Same work, 32x
// shorter dependent chain, 32x more parallelism.
// Warp layout <L, SPL>: a warp is 32/L groups of L lanes; every group owns SPL seeds and its L lanes
// share the sweep (lane j of the group takes point pairs j, j+L, ...).  Seeds per warp = 32/L * SPL:
//   <4,2> = 16 seeds: lanes of different groups read the SAME point pair (shared-memory broadcast), so
//           a sweep step costs 2 wavefronts instead of 16 -- the throughput layout while thousands of
//           seeds are left;
//   <32,1> = 1 seed: the shortest dependent chain (n_c/64 steps) -- the latency layout for the last,
//           nearly empty phases.
template <int L, int SPL>
__device__ __forceinline__ void ms_run_tile_split(const MsArgs &a, MsIterSmem &sm, int f, int tile,
                                                  int it_lo, int it_hi, int cur, int nxt,
                                                  int warps_live = kMsWarps) {
  constexpr int kGroups = 32 / L;
  constexpr int kSeedsPerWarp = kGroups * SPL;
  const int start = a.fit_start[f], n_c = a.fit_count[f];
  const int n_act = a.act_cnt[static_cast<size_t>(cur) * a.n_fits + f];
  const int *act_cur = a.act + static_cast<size_t>(cur) * a.cap + start;
  int *act_nxt = a.act + static_cast<size_t>(nxt) * a.cap + start;
  const int t = threadIdx.x;
  const unsigned lane = t & 31u, warp = t >> 5;
  const int grp = static_cast<int>(lane) / L, sub = static_cast<int>(lane) % L;
  const float k = a.kexp;
  const bool single = n_c <= kMsPtTile;
  const bool freeze_on = !(a.flags & PVN3D_MS_NO_FREEZE);
  const int star = a.max_idx[f];

  __syncthreads();
  if (single) {
    ms_stage_pairs(sm.pts, a.cpts + start, n_c);
    __syncthreads();
  }
  int idx[SPL];
  float cx[SPL], cy[SPL], cz[SPL], last[SPL];
  bool frozen[SPL];
#pragma unroll
  for (int r = 0; r < SPL; ++r) {
    const int pos = (tile * warps_live + static_cast<int>(warp)) * kSeedsPerWarp + r * kGroups + grp;
    const bool valid = static_cast<int>(warp) < warps_live && pos < n_act;
    idx[r] = valid ? act_cur[pos] : -1;
    const float4 c = a.seeds[start + (valid ? idx[r] : 0)];
    cx[r] = c.x; cy[r] = c.y; cz[r] = c.z; last[r] = c.w;
    frozen[r] = !valid;
  }
  for (int it = it_lo; it <= it_hi; ++it) {
    bool mine_frozen = true;
#pragma unroll
    for (int r = 0; r < SPL; ++r) mine_frozen &= frozen[r];
    const bool warp_live = !__all_sync(0xffffffffu, mine_frozen);
    if (single && !warp_live) break;
    MsSeedQ sq[SPL];
    MsSeedS ss[SPL];
#pragma unroll
    for (int r = 0; r < SPL; ++r) {
      sq[r] = ms_seed_q(k, cx[r], cy[r], cz[r]);
      ss[r].sw = ss[r].sx = ss[r].sy = ss[r].sz = make_float2(0.f, 0.f);
    }
    for (int base = 0; base < n_c; base += kMsPtTile) {
      const int n = min(kMsPtTile, n_c - base);
      if (!single) {
        __syncthreads();
        ms_stage_pairs(sm.pts, a.cpts + start + base, n);
        __syncthreads();
      }
      if (warp_live) {
        const int npairs = (n + 1) >> 1;
#pragma unroll 4
        for (int p = sub; p < npairs; p += L) {
          const float4 A = sm.pts[p], B = sm.pts[kMsPairs + p];
#pragma unroll
          for (int r = 0; r < SPL; ++r) ms_pair_step(A, B, sq[r], ss[r]);
        }
      }
    }
    float sw[SPL], sx[SPL], sy[SPL], sz[SPL];
#pragma unroll
    for (int r = 0; r < SPL; ++r) {
      sw[r] = ss[r].sw.x + ss[r].sw.y;
      sx[r] = ss[r].sx.x + ss[r].sx.y;
      sy[r] = ss[r].sy.x + ss[r].sy.y;
      sz[r] = ss[r].sz.x + ss[r].sz.y;
    }
#pragma unroll
    for (int o = L / 2; o > 0; o >>= 1) {  // butterfly inside the group: every lane gets the totals
#pragma unroll
      for (int r = 0; r < SPL; ++r) {
        sw[r] += __shfl_xor_sync(0xffffffffu, sw[r], o);
        sx[r] += __shfl_xor_sync(0xffffffffu, sx[r], o);
        sy[r] += __shfl_xor_sync(0xffffffffu, sy[r], o);
        sz[r] += __shfl_xor_sync(0xffffffffu, sz[r], o);
      }
    }
    bool violates = false;
#pragma unroll
    for (int r = 0; r < SPL; ++r) {
      if (!frozen[r]) {
        const float nx = __fdiv_rn(sx[r], sw[r]), ny = __fdiv_rn(sy[r], sw[r]),
                    nz = __fdiv_rn(sz[r], sw[r]);
        const float sh = __fsqrt_rn(torch_sqnorm(nx - cx[r], ny - cy[r], nz - cz[r]));
        cx[r] = nx; cy[r] = ny; cz[r] = nz; last[r] = sh;
        violates |= !(sh < a.stop_thresh);
        const bool still = sh < a.eps_stat;
        if (idx[r] == star && sub == 0) {
          a.traj[static_cast<size_t>(f) * a.traj_stride + it] = make_float4(nx, ny, nz, sh);
          if (still && a.star_it[f] == 0) a.star_it[f] = it;
        }
        if (still && freeze_on) frozen[r] = true;
      }
    }
    if (__any_sync(0xffffffffu, violates) && lane == 0)
      atomicOr(a.viol + static_cast<size_t>(f) * a.viol_words + (it >> 5), 1u << (it & 31));
    if (!single) {
      bool fr = true;
#pragma unroll
      for (int r = 0; r < SPL; ++r) fr &= frozen[r];
      if (!__syncthreads_or(fr ? 0 : 1)) break;
    }
  }
  if (sub == 0) {
#pragma unroll
    for (int r = 0; r < SPL; ++r) {
      if (idx[r] >= 0) {
        a.seeds[start + idx[r]] = make_float4(cx[r], cy[r], cz[r], last[r]);
        if (!frozen[r]) {
          const int at = atomicAdd(a.act_cnt + static_cast<size_t>(nxt) * a.n_fits + f, 1);
          act_nxt[at] = idx[r];
        }
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------
// PVN3D_MS_CERTIFIED: the fit's answer from ~32 seeds instead of n_c.
//
// fit() returns C[max_idx] after T iterations, T being the first iteration at which NO seed moves by
// >= bw*1e-3.  The returned seed ("star", the densest input) sits in the cluster and is stationary
// after s ~ 4-10 iterations, while T on votes with outliers is 60-300 -- the creeping outlier seeds
// set it, and sweeping them is n_c^2 pair evaluations per iteration for a number nobody reads.
// One CTA per fit:
//   1. iterate the star until its shift is < 1e-6*bw (iteration s); it0 = the first iteration from
//      which its remaining path length to C_s is below delta = 1e-5*bw;
//   2. alongside, iterate 31 WITNESS seeds (per residue class of the index: the input farthest from
//      the star; second pool: the input with the lowest density count) and record at which iterations
//      one of them still moves by >= bw*1e-3;
//   3. if every iteration it < it0 has such a witness, the reference's rule cannot have fired before
//      it0 (its maximum runs over ALL seeds, the witnesses included): T >= it0, and therefore
//      |C_T - C_s| < delta (T <= s: remaining path; T > s: drift of a stationary seed).  The fit is
//      marked done (= 2), ctr = C_s, ctr.w = it0.
//   4. otherwise the fit is left to ms_iterate_kernel (all seeds, reference rule + early exit).
// Witnesses only ever ADD evidence (a violation observed is a violation of the full sweep, since a
// seed's trajectory depends on nothing but itself and the fixed points), so a bad witness choice costs
// time (fallback), never correctness.
constexpr int kWitSlots = 32;            // seeds per pool: 8 warps x 4
constexpr int kWitPerWarp = kWitSlots / kMsWarps;
constexpr int kWitPools = 2;
constexpr int kWitViolWords = 128;       // max_iter <= 4094 -> iterations <= 4095

struct MsWitSmem {
  float4 pts[kMsPtTile];
  unsigned viol[kWitViolWords];
  int slot_idx[kWitSlots];
  int s_it;     // iteration at which the star became stationary (0 = not yet)
  int it0;
  int certified;
};

__global__ void __launch_bounds__(kMsThreads, 2) ms_witness_kernel(MsArgs a) {
  extern __shared__ __align__(16) unsigned char ms_smem_raw[];
  MsWitSmem &sm = *reinterpret_cast<MsWitSmem *>(ms_smem_raw);
  const int f = blockIdx.x;
  const int n_c = a.fit_count[f];
  if (n_c <= 0) return;
  const int start = a.fit_start[f], star = a.max_idx[f];
  const int last_it = a.max_iter + 1;
  const bool single = n_c <= kMsPtTile;
  const int t = threadIdx.x;
  const unsigned lane = t & 31u;
  const int warp = t >> 5;
  const float k = a.kexp;
  const float4 *cpts = a.cpts + start;

  if (single) ms_stage_pairs(sm.pts, cpts, n_c);
  for (int w = t; w < kWitViolWords; w += kMsThreads) sm.viol[w] = 0u;
  if (t == 0) { sm.s_it = 0; sm.it0 = 0; sm.certified = 0; }
  __syncthreads();

  for (int pool = 0; pool < kWitPools; ++pool) {
    // ---- the pool's seeds: slot = residue class (index mod 256) / 8 --------------------------------
    {
      float best = __int_as_float(0x7f800000);
      int besti = -1;
      for (int i = t; i < n_c; i += kMsThreads) {
        // pool 0: farthest from the star (cpts.w = k |a'|^2, k < 0: the smallest value is the farthest);
        // pool 1: lowest density count
        const float key = pool == 0 ? cpts[i].w : static_cast<float>(a.dens_cnt[start + i]);
        if (key < best) { best = key; besti = i; }
      }
#pragma unroll
      for (int o = 4; o > 0; o >>= 1) {
        const float ob = __shfl_xor_sync(0xffffffffu, best, o);
        const int oi = __shfl_xor_sync(0xffffffffu, besti, o);
        if (oi >= 0 && (besti < 0 || ob < best || (ob == best && oi < besti))) { best = ob; besti = oi; }
      }
      if ((t & 7) == 0) sm.slot_idx[t >> 3] = (pool == 0 && t == 0) ? star : besti;
    }
    __syncthreads();
    const int it_hi = pool == 0 ? last_it : sm.it0 - 1;   // later pools only need marks below it0

    int idx[kWitPerWarp];
    float cx[kWitPerWarp], cy[kWitPerWarp], cz[kWitPerWarp];
    bool frozen[kWitPerWarp];
#pragma unroll
    for (int r = 0; r < kWitPerWarp; ++r) {
      idx[r] = sm.slot_idx[warp * kWitPerWarp + r];
      const float4 c = cpts[idx[r] >= 0 ? idx[r] : 0];
      cx[r] = c.x; cy[r] = c.y; cz[r] = c.z;
      frozen[r] = idx[r] < 0;
    }
    const bool has_star = pool == 0 && warp == 0;   // slot 0 of pool 0

    // evidence must survive the ~1e-6 relative difference between this arithmetic and the reference's:
    // a witness counts only when it moves by 1 % more than the threshold
    const float wit_thresh = a.stop_thresh * 1.01f;
    for (int it = 1; it <= it_hi; ++it) {
      bool star_still = false;
      bool warp_live = false;
#pragma unroll
      for (int r = 0; r < kWitPerWarp; ++r) warp_live |= !frozen[r];   // uniform across the warp
      MsSeedQ sq[kWitPerWarp];
      MsSeedS ss[kWitPerWarp];
#pragma unroll
      for (int r = 0; r < kWitPerWarp; ++r) {
        sq[r] = ms_seed_q(k, cx[r], cy[r], cz[r]);
        ss[r].sw = ss[r].sx = ss[r].sy = ss[r].sz = make_float2(0.f, 0.f);
      }
      for (int base = 0; base < n_c; base += kMsPtTile) {
        const int n = min(kMsPtTile, n_c - base);
        if (!single) {
          __syncthreads();
          ms_stage_pairs(sm.pts, cpts + base, n);
          __syncthreads();
        }
        if (warp_live) {
          const int npairs = (n + 1) >> 1;
#pragma unroll 2
          for (int p = lane; p < npairs; p += 32) {
            const float4 A = sm.pts[p], B = sm.pts[kMsPairs + p];
#pragma unroll
            for (int r = 0; r < kWitPerWarp; ++r) ms_pair_step(A, B, sq[r], ss[r]);
          }
        }
      }
      if (warp_live) {
        float sw[kWitPerWarp], sx[kWitPerWarp], sy[kWitPerWarp], sz[kWitPerWarp];
#pragma unroll
        for (int r = 0; r < kWitPerWarp; ++r) {
          sw[r] = ss[r].sw.x + ss[r].sw.y;
          sx[r] = ss[r].sx.x + ss[r].sx.y;
          sy[r] = ss[r].sy.x + ss[r].sy.y;
          sz[r] = ss[r].sz.x + ss[r].sz.y;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
          for (int r = 0; r < kWitPerWarp; ++r) {
            sw[r] += __shfl_xor_sync(0xffffffffu, sw[r], o);
            sx[r] += __shfl_xor_sync(0xffffffffu, sx[r], o);
            sy[r] += __shfl_xor_sync(0xffffffffu, sy[r], o);
            sz[r] += __shfl_xor_sync(0xffffffffu, sz[r], o);
          }
        }
        bool violates = false;
#pragma unroll
        for (int r = 0; r < kWitPerWarp; ++r) {
          if (!frozen[r]) {
            const float nx = __fdiv_rn(sx[r], sw[r]), ny = __fdiv_rn(sy[r], sw[r]),
                        nz = __fdiv_rn(sz[r], sw[r]);
            const float sh = __fsqrt_rn(torch_sqnorm(nx - cx[r], ny - cy[r], nz - cz[r]));
            cx[r] = nx; cy[r] = ny; cz[r] = nz;
            violates |= !(sh < wit_thresh);
            const bool still = sh < a.eps_stat;
            if (has_star && r == 0 && lane == 0) {
              a.traj[static_cast<size_t>(f) * a.traj_stride + it] = make_float4(nx, ny, nz, sh);
              if (still) { sm.s_it = it; star_still = true; }
            }
            if (still) frozen[r] = true;
          }
        }
        if (violates && lane == 0) atomicOr(&sm.viol[it >> 5], 1u << (it & 31));
      }
      // block-uniform: the star is stationary -- nothing after s is needed
      if (__syncthreads_or(star_still ? 1 : 0)) break;
    }

    // ---- verdict after this pool (thread 0; every value it reads it wrote itself or is in smem) ----
    if (t == 0) {
      const int s_it = sm.s_it;
      if (s_it > 0) {
        if (pool == 0) {
          float acc = 0.f;
          int it0 = s_it;
          for (int j = s_it; j >= 1; --j) {
            acc += a.traj[static_cast<size_t>(f) * a.traj_stride + j].w;
            if (!(acc < a.delta_path)) break;
            it0 = j - 1;
          }
          sm.it0 = max(it0, 1);
        }
        bool ok = true;
        for (int it = 1; it < sm.it0; ++it)
          if (!((sm.viol[it >> 5] >> (it & 31)) & 1u)) { ok = false; break; }
        sm.certified = ok ? 1 : 0;
      }
    }
    __syncthreads();
    if (sm.s_it == 0 || sm.certified) break;   // no stationary star within max_iter, or done
  }

  if (t == 0 && sm.certified) {
    const float4 c = a.traj[static_cast<size_t>(f) * a.traj_stride + sm.s_it];
    const float4 o = a.pts[start + star];
    a.ctr[f] = make_float4(c.x + o.x, c.y + o.y, c.z + o.z, static_cast<float>(sm.it0));
    a.iters[f] = sm.it0;
    a.star_it[f] = sm.s_it;
    a.done[f] = 2;
    atomicAdd(a.cfg + kMsCfgCertified, 1);   // statistics: fits certified by this launch
  }
}

// ------------------------------------------------------------------------------------------------
// Fallback of PVN3D_MS_CERTIFIED: the fits the witnesses could not close (typically clean vote sets whose
// global stop rule fires within a few iterations) are iterated over ALL seeds by ONE CTA per fit, in lock
// step like the reference loop, with the rule of PVN3D_MS_EARLY_EXIT: stop at the first iteration at which no
// seed moves by >= bw*1e-3 (the reference's T), or at which the returned seed is stationary.  Seeds that
// stopped moving (< 1e-6*bw) are skipped like in ms_iterate_kernel.
// Unlike ms_iterate_kernel this is an ordinary launch: no grid barrier, no co-residency requirement -- a
// cooperative grid of 3 CTAs on EVERY SM cannot start while the persistent MLP kernels of hot path A and the
// sampling CTAs of the look-ahead stream hold SMs, and would serialise the streams of the frame pipeline.
struct MsFbSmem {
  float4 pts[kMsPtTile];
  int violated[3];   // flag of iteration it lives in slot it % 3; slot (it+1) % 3 is cleared during iteration it
                     // (last read at the end of iteration it-2, a barrier ago)
  int star_still;
  float4 star_pos;
};

__global__ void __launch_bounds__(kMsThreads, 3) ms_fallback_kernel(MsArgs a) {
  extern __shared__ __align__(16) unsigned char ms_smem_raw[];
  MsFbSmem &sm = *reinterpret_cast<MsFbSmem *>(ms_smem_raw);
  const int f = blockIdx.x;
  const int n_c = a.fit_count[f];
  if (n_c <= 0 || a.done[f]) return;   // empty, or certified
  const int start = a.fit_start[f], star = a.max_idx[f];
  const int last_it = a.max_iter + 1;
  const bool single = n_c <= kMsPtTile;
  const int t = threadIdx.x;
  const float k = a.kexp;
  const float4 *cpts = a.cpts + start;
  float4 *seeds = a.seeds + start;
  constexpr int R = 2;
  if (single) ms_stage_pairs(sm.pts, cpts, n_c);
  if (t == 0) { sm.violated[0] = sm.violated[1] = sm.violated[2] = 0; sm.star_still = 0; sm.star_pos = make_float4(0.f, 0.f, 0.f, 0.f); }
  __syncthreads();
  int T = last_it;
  for (int it = 1; it <= last_it; ++it) {
    if (t == 0) sm.violated[(it + 1) % 3] = 0;
    for (int base = 0; base < n_c; base += kMsThreads * R) {
      int idx[R];
      float cx[R], cy[R], cz[R];
      bool skip[R];
      bool any = false;
#pragma unroll
      for (int r = 0; r < R; ++r) {
        idx[r] = base + r * kMsThreads + t;
        const bool valid = idx[r] < n_c;
        const float4 c = seeds[valid ? idx[r] : 0];
        cx[r] = c.x; cy[r] = c.y; cz[r] = c.z;
        skip[r] = !valid || (it > 1 && c.w < a.eps_stat);   // .w = shift of the previous iteration
        any |= !skip[r];
      }
      const bool warp_live = __any_sync(0xffffffffu, any);
      MsSeedQ sq[R];
      MsSeedS ss[R];
#pragma unroll
      for (int r = 0; r < R; ++r) {
        sq[r] = ms_seed_q(k, cx[r], cy[r], cz[r]);
        ss[r].sw = ss[r].sx = ss[r].sy = ss[r].sz = make_float2(0.f, 0.f);
      }
      if (single) {
        if (warp_live) ms_sweep<R>(sm.pts, (n_c + 1) >> 1, sq, ss);
      } else {
        for (int pb = 0; pb < n_c; pb += kMsPtTile) {
          const int n = min(kMsPtTile, n_c - pb);
          __syncthreads();
          ms_stage_pairs(sm.pts, cpts + pb, n);
          __syncthreads();
          if (warp_live) ms_sweep<R>(sm.pts, (n + 1) >> 1, sq, ss);
        }
      }
      bool violates = false;
#pragma unroll
      for (int r = 0; r < R; ++r) {
        if (!skip[r]) {
          const float swr = ss[r].sw.x + ss[r].sw.y;
          const float nx = __fdiv_rn(ss[r].sx.x + ss[r].sx.y, swr), ny = __fdiv_rn(ss[r].sy.x + ss[r].sy.y, swr),
                      nz = __fdiv_rn(ss[r].sz.x + ss[r].sz.y, swr);
          const float sh = __fsqrt_rn(torch_sqnorm(nx - cx[r], ny - cy[r], nz - cz[r]));
          seeds[idx[r]] = make_float4(nx, ny, nz, sh);
          violates |= !(sh < a.stop_thresh);
          if (idx[r] == star) {
            sm.star_pos = make_float4(nx, ny, nz, sh);
            if (sh < a.eps_stat) sm.star_still = 1;
          }
        }
      }
      if (__any_sync(0xffffffffu, violates) && (t & 31) == 0) sm.violated[it % 3] = 1;
    }
    __syncthreads();
    const bool viol = sm.violated[it % 3] != 0, still = sm.star_still != 0;
    if (!viol || still) { T = it; break; }   // the reference's T, or the returned seed is stationary (block-uniform)
  }
  if (t == 0) {
    // the star's latest position is C after exactly T iterations (every seed is swept at iteration 1)
    const float4 c = sm.star_pos;
    const float4 o = a.pts[start + star];
    a.ctr[f] = make_float4(c.x + o.x, c.y + o.y, c.z + o.z, static_cast<float>(T));
    a.iters[f] = T;
    a.done[f] = 1;
  }
}

__global__ void __launch_bounds__(kMsThreads, 3) ms_iterate_kernel(MsArgs a) {
  extern __shared__ __align__(16) unsigned char ms_smem_raw[];
  MsIterSmem &sm = *reinterpret_cast<MsIterSmem *>(ms_smem_raw);
  unsigned epoch = 0;
  unsigned *gbar = reinterpret_cast<unsigned *>(a.cfg + 3);  // zeroed by ms_setup_kernel
  const int t = threadIdx.x;
  const int per_thread = (a.n_fits + kMsThreads - 1) / kMsThreads;  // <= 8
  const int f_lo = min(a.n_fits, t * per_thread), f_hi = min(a.n_fits, f_lo + per_thread);
  const int last_it = a.max_iter + 1;  // the reference breaks when it > max_iter (:42)
  const bool early = a.flags & PVN3D_MS_EARLY_EXIT;
  // rank of this CTA among the CTAs resident on its SM: phases with few tiles hand them to rank 0
  // first, so that the tiles land on DIFFERENT SMs (a tile is bound by its SM's MUFU / LDS rate)
  if (t == 0) {
    unsigned smid;
    asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
    sm.ticket = atomicAdd(a.cfg + kMsCfgSm + static_cast<int>(smid & 1023u), 1);
  }
  __syncthreads();
  const int sm_rank = sm.ticket;
  const int n_sm = max(1, static_cast<int>(gridDim.x) / max(1, a.ctas_per_sm));
  __syncthreads();

  for (int p = 0;; ++p) {
    const int cur = p % 3, nxt = (p + 1) % 3, nxt2 = (p + 2) % 3;
    const int prev_lo = p > 0 ? (p > 1 ? ms_phase_end(p - 2) + 1 : 1) : 0;
    const int prev_hi = p > 0 ? min(ms_phase_end(p - 1), last_it) : 0;
    const int it_lo = prev_hi + 1, it_hi = min(ms_phase_end(p), last_it);

    // ---- per-fit decisions on the finished phase (identical in every CTA) ---------------------
    int local_seeds = 0;
    for (int f = f_lo; f < f_hi; ++f) {
      int dn = a.done[f];
      const int n_act = a.act_cnt[static_cast<size_t>(cur) * a.n_fits + f];
      if (!dn && p > 0) {
        int tz = 0;
        const unsigned *vw = a.viol + static_cast<size_t>(f) * a.viol_words;
        for (int it = prev_lo; it <= prev_hi; ++it)
          if (!((vw[it >> 5] >> (it & 31)) & 1u)) { tz = it; break; }
        // CTAs that are through with these decisions already run tiles of phase p, which may set star_it
        // to an iteration of phase p; only a value from a finished phase keeps the decision identical in
        // every CTA (a CTA that alone closed the fit could leave the loop while the others wait at the barrier)
        int s = a.star_it[f];
        if (s > prev_hi) s = 0;
        int T = 0;
        if (tz) T = (early && s > 0 && s < tz) ? s : tz;
        else if (early && s > 0) T = s;
        else if (prev_hi >= last_it) T = last_it;
        else if (n_act == 0) T = prev_hi;  // cannot happen (an all-frozen fit clears a bit); safe exit
        if (T) {
          dn = 1;
          a.done[f] = 1;  // every CTA derives the same value from the same data
          a.iters[f] = T;
        }
      }
      a.act_cnt[static_cast<size_t>(nxt2) * a.n_fits + f] = 0;  // list of phase p+2, idle since p-1
      sm.prefix[f] = dn ? 0 : n_act;
      local_seeds += dn ? 0 : n_act;
    }
    int total_seeds;
    (void)block_exclusive_scan<kMsThreads>(local_seeds, sm.warp_scan, &total_seeds);
    if (total_seeds == 0 || it_lo > last_it) break;  // identical in every CTA
    // seeds per thread: keep >= 2 tiles per CTA of the grid when there is enough work; with less than
    // one full tile per CTA left, switch to the split sweep (a warp per pair of seeds)
    int R = 2;
    if (total_seeds / (kMsThreads * R) < 2 * static_cast<int>(gridDim.x)) R = 1;
    const bool split = total_seeds < kMsThreads * static_cast<int>(gridDim.x);
    // split sweep: seeds per warp (16, 8, 4, 2, 1) -- as many as keeps every warp of the grid busy
    const int warps_total = kMsWarps * static_cast<int>(gridDim.x);
    int spw = 16;
    while (spw > 1 && total_seeds < spw * warps_total) spw >>= 1;
    // ... or up to 4x fewer, if that fills the last round of tiles better: tiles cost the same, so a
    // phase takes ceil(tiles / CTAs) rounds of (spw + staging) -- 624 tiles on 444 CTAs waste 30 %
    if (split && spw >= 2) {
      int best = spw;
      long long best_cost = 0x7fffffffffffffffll;
      for (int c = spw; c >= 1 && c * 4 >= spw; c >>= 1) {
        int lt = 0;
        for (int f = f_lo; f < f_hi; ++f) lt += (sm.prefix[f] + kMsWarps * c - 1) / (kMsWarps * c);
        int tiles_c;
        (void)block_exclusive_scan<kMsThreads>(lt, sm.warp_scan, &tiles_c);
        const long long rounds = (tiles_c + static_cast<int>(gridDim.x) - 1) / static_cast<int>(gridDim.x);
        const long long cost = rounds * (c + 1);
        if (cost < best_cost) { best_cost = cost; best = c; }
      }
      spw = best;
    }
    // last phases: fewer seeds than warps on one CTA per SM -> smaller tiles (1, 2 or 4 live warps)
    int warps_live = kMsWarps;
    if (split && spw == 1)
      while (warps_live > 1 && total_seeds < warps_live * n_sm) warps_live >>= 1;
    const int tile_seeds = split ? warps_live * spw : kMsThreads * R;
    int local_tiles = 0;
    for (int f = f_lo; f < f_hi; ++f) local_tiles += (sm.prefix[f] + tile_seeds - 1) / tile_seeds;
    int total;
    int excl = block_exclusive_scan<kMsThreads>(local_tiles, sm.warp_scan, &total);
    for (int f = f_lo; f < f_hi; ++f) {
      const int tiles = (sm.prefix[f] + tile_seeds - 1) / tile_seeds;
      sm.prefix[f] = excl;
      excl += tiles;
    }
    if (t == 0) sm.prefix[a.n_fits] = total;
    __syncthreads();
    if (blockIdx.x == 0 && t == 0) a.cfg[nxt] = 0;  // ticket counter of the next phase
    if ((a.flags & 4u) && blockIdx.x == 0 && t == 0 && p < 60) {  // PVN3D_MS_DEBUG_TIMING: stamps in cfg
      unsigned long long ns;
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(ns));
      a.cfg[16 + p] = static_cast<int>((ns / 1000ull) & 0x3fffffffull);  // top of phase p (us)
      a.cfg[136 + p] = total_seeds;
      a.cfg[196 + p] = total;
    }

    // ---- tiles of this phase, handed out dynamically -------------------------------------------
    const bool takes_tiles = static_cast<long long>(sm_rank) * n_sm < total;
    for (; takes_tiles;) {
      if (t == 0) sm.ticket = atomicAdd(a.cfg + cur, 1);
      __syncthreads();
      const int tk = sm.ticket;
      __syncthreads();
      if (tk >= total) break;
      const int f = find_segment(sm.prefix, a.n_fits, tk);
      const int tile = tk - sm.prefix[f];
      if (split && spw == 16) ms_run_tile_split<4, 2>(a, sm, f, tile, it_lo, it_hi, cur, nxt);
      else if (split && spw == 8) ms_run_tile_split<8, 2>(a, sm, f, tile, it_lo, it_hi, cur, nxt);
      else if (split && spw == 4) ms_run_tile_split<16, 2>(a, sm, f, tile, it_lo, it_hi, cur, nxt);
      else if (split && spw == 2) ms_run_tile_split<32, 2>(a, sm, f, tile, it_lo, it_hi, cur, nxt);
      else if (split) ms_run_tile_split<32, 1>(a, sm, f, tile, it_lo, it_hi, cur, nxt, warps_live);
      else if (R == 2) ms_run_tile<2>(a, sm, f, tile, it_lo, it_hi, cur, nxt);
      else ms_run_tile<1>(a, sm, f, tile, it_lo, it_hi, cur, nxt);
    }
    if ((a.flags & 4u) && t == 0) {
      unsigned long long ns;
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(ns));
      if (p < 60) atomicMax(a.cfg + 76 + p, static_cast<int>((ns / 1000ull) & 0x3fffffffull));  // tiles done
    }
    ms_grid_barrier(gbar, epoch);
  }

  // ---- results: C[max_idx] after exactly T iterations, back in world coordinates (:51) -----------
  for (int f = blockIdx.x * kMsThreads + t; f < a.n_fits; f += gridDim.x * kMsThreads) {
    const int cnt = a.fit_count[f];
    if (cnt <= 0 || a.done[f] == 2) continue;  // empty, or certified (ms_witness_kernel wrote ctr)
    const int start = a.fit_start[f], mi = a.max_idx[f];
    const int T = a.iters[f], s = a.star_it[f];
    const bool frozen_before_T = !(a.flags & PVN3D_MS_NO_FREEZE) && s > 0 && T >= s;
    const float4 c = frozen_before_T ? a.seeds[start + mi]
                                     : a.traj[static_cast<size_t>(f) * a.traj_stride + T];
    const float4 o = a.pts[start + mi];
    a.ctr[f] = make_float4(c.x + o.x, c.y + o.y, c.z + o.z, static_cast<float>(T));
  }
}

// smallest float t2 such that sqrtf(t2) >= bwf  =>  (sqrtf(d2) < bwf) == (d2 < t2) for all d2 >= 0
float density_threshold(float bwf) {
  if (!(bwf > 0.f)) return 0.f;  // nothing is < 0
  float t = bwf * bwf;
  while (sqrtf(t) >= bwf && t > 0.f) t = nextafterf(t, 0.f);
  while (sqrtf(t) < bwf) t = nextafterf(t, INFINITY);
  return t;
}

struct MsLayout {
  size_t cpts, seeds, best_key, done, iters, star, act, act_cnt, viol, traj, dens_prefix, dens_cnt, cfg, total;
  int viol_words, traj_stride;
};
MsLayout ms_layout(int cap, int n_fits, int max_iter) {
  MsLayout L;
  size_t off = 0;
  auto take = [&](size_t bytes) {
    const size_t at = off;
    off = align_up(off + bytes, 256);
    return at;
  };
  const size_t nf = n_fits > 0 ? n_fits : 1, cp = cap > 0 ? cap : 1;
  L.cfg = take(kMsCfgInts * sizeof(int));  // first: debug stamps are read back from the head of the workspace
  L.cpts = take(cp * sizeof(float4));
  L.seeds = take(cp * sizeof(float4));
  L.viol_words = (max_iter + 2 + 31) / 32;
  L.traj_stride = max_iter + 2;
  L.best_key = take(nf * sizeof(unsigned long long));
  L.done = take(nf * sizeof(int));
  L.iters = take(nf * sizeof(int));
  L.star = take(nf * sizeof(int));
  L.act = take(3 * cp * sizeof(int));
  L.act_cnt = take(3 * nf * sizeof(int));
  L.viol = take(nf * L.viol_words * sizeof(unsigned));
  L.traj = take(nf * static_cast<size_t>(L.traj_stride) * sizeof(float4));
  L.dens_prefix = take((nf + 1) * sizeof(int));
  L.dens_cnt = take(cp * sizeof(int));
  L.total = off;
  return L;
}

int ms_persistent_grid(int *out, int *ctas_per_sm) {
  static int cached[64] = {0}, cached_per_sm[64] = {0};
  int dev = 0;
  PVN3D_CUDA_TRY(cudaGetDevice(&dev), "cudaGetDevice");
  if (dev >= 0 && dev < 64 && cached[dev] > 0) {
    *out = cached[dev];
    *ctas_per_sm = cached_per_sm[dev];
    return PVN3D_OK;
  }
  PVN3D_CUDA_TRY(cudaFuncSetAttribute(ms_iterate_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      (int)sizeof(MsIterSmem)),
                 "ms_iterate smem attr");
  int per_sm = 0, sms = 0;
  PVN3D_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, ms_iterate_kernel,
                                                               kMsThreads, sizeof(MsIterSmem)),
                 "ms_iterate occupancy");
  PVN3D_CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev), "sm count");
  if (per_sm < 1 || sms < 1) return PVN3D_ERR_UNSUPPORTED;
  *out = per_sm * sms;
  *ctas_per_sm = per_sm;
  if (dev >= 0 && dev < 64) {
    cached_per_sm[dev] = per_sm;
    cached[dev] = *out;
  }
  return PVN3D_OK;
}

}  // namespace

// internal entry shared with poses.cu: fits already described on device, workspace carved by caller
// density_only: stop after the exact pass (max_idx, n_in, labels); no iterations, ctr untouched
int meanshift_launch(const float4 *pts, const int *fit_start, const int *fit_count, int n_fits,
                     int cap, double bandwidth, int max_iter, unsigned flags, float4 *ctr,
                     uint8_t *labels, int *max_idx, int *n_in, unsigned char *ws, cudaStream_t st,
                     bool density_only) {
  if (n_fits <= 0) return PVN3D_OK;
  int grid = 0, per_sm = 1;
  int rc = ms_persistent_grid(&grid, &per_sm);
  if (rc != PVN3D_OK) return rc;
  const float bwf = static_cast<float>(bandwidth);
  const MsLayout L = ms_layout(cap, n_fits, max_iter);
  for (int f0 = 0; f0 < n_fits; f0 += kMsFitMax) {
    const int nf = std::min(kMsFitMax, n_fits - f0);
    MsArgs a;
    a.pts = pts;
    a.fit_start = fit_start + f0;
    a.fit_count = fit_count + f0;
    a.n_fits = nf;
    a.t2 = density_threshold(bwf);
    a.stop_thresh = static_cast<float>(bandwidth * 1e-3);
    a.eps_stat = static_cast<float>(bandwidth * 1e-6);
    a.kexp = static_cast<float>(-1.4426950408889634 / (2.0 * bandwidth * bandwidth));
    a.max_iter = max_iter;
    a.flags = flags;
    a.ctr = ctr + f0;
    a.labels = labels;
    a.max_idx = max_idx + f0;
    a.n_in = n_in + f0;
    a.cpts = reinterpret_cast<float4 *>(ws + L.cpts);
    a.seeds = reinterpret_cast<float4 *>(ws + L.seeds);
    a.best_key = reinterpret_cast<unsigned long long *>(ws + L.best_key) + f0;
    a.done = reinterpret_cast<int *>(ws + L.done) + f0;
    a.iters = reinterpret_cast<int *>(ws + L.iters) + f0;
    a.star_it = reinterpret_cast<int *>(ws + L.star) + f0;
    a.act = reinterpret_cast<int *>(ws + L.act);
    a.act_cnt = reinterpret_cast<int *>(ws + L.act_cnt) + 3 * static_cast<size_t>(f0);
    a.viol = reinterpret_cast<unsigned *>(ws + L.viol) + static_cast<size_t>(f0) * L.viol_words;
    a.traj = reinterpret_cast<float4 *>(ws + L.traj) + static_cast<size_t>(f0) * L.traj_stride;
    a.dens_prefix = reinterpret_cast<int *>(ws + L.dens_prefix);
    a.dens_cnt = reinterpret_cast<int *>(ws + L.dens_cnt);
    a.delta_path = static_cast<float>(bandwidth * 1e-5);
    a.cfg = reinterpret_cast<int *>(ws + L.cfg);
    a.cap = cap;
    a.viol_words = L.viol_words;
    a.traj_stride = L.traj_stride;
    a.ctas_per_sm = per_sm;

    ms_setup_kernel<<<1, 1024, 0, st>>>(a);
    if ((rc = check_launch("ms_setup_kernel")) != PVN3D_OK) return rc;
    // upper bound on density tiles: every fit wastes < 1 tile
    const int tiles = ceil_div(cap, kMsThreads) + nf;
    static const bool prune_env = [] { const char *e = getenv("PVN3D_MS_PRUNED_DENSITY"); return !(e && e[0] == '0'); }();
    a.dens_pruned = (prune_env && !(flags & PVN3D_MS_BRUTE_DENSITY)) ? 1 : 0;
    a.bwf = bwf;
    if (a.dens_pruned) {
      static PerDeviceOnce once_pr;
      PVN3D_ONCE_PER_DEVICE(once_pr,
                            cudaFuncSetAttribute(ms_density_pruned_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                                 (int)sizeof(MsPruneSmem)),
                            "ms_density_pruned smem attr");
      ms_density_pruned_kernel<<<nf, kMsThreads, sizeof(MsPruneSmem), st>>>(a);
      if ((rc = check_launch("ms_density_pruned_kernel")) != PVN3D_OK) return rc;
    }
    ms_density_kernel<<<tiles, kMsThreads, 0, st>>>(a);   // fits above kMsPruneMax points (all fits without pruning)
    if ((rc = check_launch("ms_density_kernel")) != PVN3D_OK) return rc;
    ms_prepare_kernel<<<tiles, kMsThreads, 0, st>>>(a);
    if ((rc = check_launch("ms_prepare_kernel")) != PVN3D_OK) return rc;
    if (density_only) continue;
    if (flags & PVN3D_MS_CERTIFIED) {
      static PerDeviceOnce once;
      PVN3D_ONCE_PER_DEVICE(once,
                            cudaFuncSetAttribute(ms_witness_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                                 (int)sizeof(MsWitSmem)),
                            "ms_witness smem attr");
      ms_witness_kernel<<<nf, kMsThreads, sizeof(MsWitSmem), st>>>(a);
      if ((rc = check_launch("ms_witness_kernel")) != PVN3D_OK) return rc;
      static PerDeviceOnce once_fb;
      PVN3D_ONCE_PER_DEVICE(once_fb,
                            cudaFuncSetAttribute(ms_fallback_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                                 (int)sizeof(MsFbSmem)),
                            "ms_fallback smem attr");
      ms_fallback_kernel<<<nf, kMsThreads, sizeof(MsFbSmem), st>>>(a);
      if ((rc = check_launch("ms_fallback_kernel")) != PVN3D_OK) return rc;
      continue;   // no cooperative launch in this mode
    }
    void *kargs[] = {&a};
    PVN3D_CUDA_TRY(cudaLaunchCooperativeKernel(reinterpret_cast<void *>(ms_iterate_kernel),
                                               dim3(grid), dim3(kMsThreads), kargs,
                                               sizeof(MsIterSmem), st),
                   "ms_iterate_kernel launch");
    count_launch();
  }
  return PVN3D_OK;
}

size_t meanshift_ws_bytes(int cap, int n_fits, int max_iter) {
  return ms_layout(cap, n_fits, max_iter).total;
}

}  // namespace pvn3d

extern "C" size_t pvn3d_meanshift_workspace_bytes(int cap, int n_fits, int max_iter) {
  if (cap < 0 || n_fits < 0 || max_iter < 0 || max_iter > 4094) return 0;
  return pvn3d::meanshift_ws_bytes(cap, n_fits, max_iter);
}

extern "C" int pvn3d_meanshift_fit_batch(const float *pts, const int *fit_start,
                                         const int *fit_count, int n_fits, int cap,
                                         double bandwidth, int max_iter, unsigned flags, float *ctr,
                                         uint8_t *labels, int *max_idx, int *n_in, void *workspace,
                                         size_t workspace_bytes, pvn3d_stream_t stream) {
  using namespace pvn3d;
  if (!pts || !fit_start || !fit_count || !ctr || !max_idx || !n_in || !workspace || n_fits < 0 ||
      cap < 0 || !(bandwidth > 0.0) || max_iter < 0)
    return PVN3D_ERR_INVALID_ARG;
  if (max_iter > 4094) return PVN3D_ERR_UNSUPPORTED;
  if (workspace_bytes < meanshift_ws_bytes(cap, n_fits, max_iter)) return PVN3D_ERR_WORKSPACE;
  if ((reinterpret_cast<uintptr_t>(pts) & 15u) || (reinterpret_cast<uintptr_t>(ctr) & 15u) ||
      (reinterpret_cast<uintptr_t>(workspace) & 255u))
    return PVN3D_ERR_INVALID_ARG;
  return meanshift_launch(reinterpret_cast<const float4 *>(pts), fit_start, fit_count, n_fits, cap,
                          bandwidth, max_iter, flags, reinterpret_cast<float4 *>(ctr), labels,
                          max_idx, n_in, static_cast<unsigned char *>(workspace),
                          pvn3d::as_stream(stream), false);
}

extern "C" size_t pvn3d_meanshift_workspace_counts_offset(int cap, int n_fits, int max_iter) {
  if (cap < 0 || n_fits < 0 || max_iter < 0 || max_iter > 4094) return 0;
  return pvn3d::ms_layout(cap, n_fits, max_iter).dens_cnt;
}
