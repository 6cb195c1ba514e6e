// Farthest-point sampling + gather for sm_100a.
//
// Replaces furthest_point_sampling_kernel<512> and gather_points_kernel (reference
// utils/sampling/fps/furthest_point_sampling.cu:99-207, :38-50) and their host wrappers
// (furthest_point_sampling.cpp:27-50, :79-100), bit for bit.
//
// What the reference computes (and this kernel reproduces exactly):
//   idx[0] = 0; temp[k] = 1e10; then m-1 times: centre = point idx[j-1]; for every point k with
//   (double)fma(z,z,fma(x,x,y*y)) > 1e-3:  temp[k] = fminf(temp[k], fma(dz,dz,fma(dx,dx,dy*dy)));
//   idx[j] = arg-max temp over those points. The reference's arg-max is a strided per-thread scan
//   (strict >) followed by a shared-memory tree that keeps the left operand on ties, so among
//   bit-equal maxima it returns the point minimising (bitreverse_L(k mod T), k div T), where
//   T = min(2^floor(log2 n), 512) is its block size and L = log2 T. With no eligible point every
//   pick is index 0.
//
// Two kernels, one CTA per cloud each:
//
// fps_pruned_kernel (n <= 32768, the path every config takes)
//   prologue  eligible points are counting-sorted by a 4096-cell grid (x,y Morton-interleaved, z low
//             bits) into a SoA copy in the L2-resident workspace, whose first 17 792 points are then
//             staged into shared memory by 1-D TMA bulk copies, so that the 128 points owned by one (warp, slot) pair form a
//             spatially tight *bucket*; each bucket keeps its bounding box and (max distance, tie
//             key, position, original index) of its current best point in shared memory;
//   loop      running distances never leave registers (64 per thread). Per iteration a lane tests
//             one bucket: LB = fma(gz,gz,fma(gx,gx,gy*gy)) on the per-axis gaps between the new
//             centre and the box. Every operation of the reference's distance is monotone in
//             |dx|,|dy|,|dz| and rounding is monotone, so LB <= d(k) for every point k of the bucket
//             *in floating point*; when LB >= the bucket's max distance no fminf can change
//             anything and the bucket is skipped -- results stay bit-identical while late
//             iterations touch only the buckets near the new centre. Touched buckets are updated
//             with packed FP32 math (sub/mul/fma.f32x2) and re-elect their best point with warp
//             REDUX; the block arg-max is a REDUX over bucket records, one smem hop across the 16
//             warps and a single __syncthreads (slots double buffered by iteration parity);
//   ties      resolved explicitly on the reference's key (bitreverse_L(k mod T), k div T).
//
// fps_flat_kernel (n > 32768, or DUSTY_FPS_FLAT=1): no pruning; points compacted in tie-break
//   order, distances in registers (or, beyond 32768 points, in the workspace).
#include <algorithm>
#include <cstdlib>

#include "common.cuh"

namespace dusty {
namespace fps {

constexpr int TPB = 512;
constexpr int NW = TPB / 32;
constexpr int GROUPS_MAX = 16;                   // 4 points per group per thread
constexpr int REG_CAP = TPB * 4 * GROUPS_MAX;    // 32768 points with register-resident distances
constexpr int SMEM_CAP = 18432;                  // points whose coordinates are staged in smem (216 KB)
constexpr int SMEM_BYTES = SMEM_CAP * 12;

__device__ __forceinline__ unsigned bitrev(unsigned v, int bits) { return bits ? (__brev(v) >> (32 - bits)) : 0u; }

struct WinSlot { unsigned val; unsigned e; };

// Block-wide exclusive scan of one int per thread (TPB threads); also returns the total.
__device__ __forceinline__ int block_exscan(int v, int* total, int* wsum) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int inc = v;
  #pragma unroll
  for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += t; }
  if (lane == 31) wsum[warp] = inc;
  __syncthreads();
  int base = 0, tot = 0;
  #pragma unroll
  for (int w = 0; w < NW; ++w) { const int s = wsum[w]; if (w < warp) base += s; tot += s; }
  __syncthreads();
  *total = tot;
  return base + inc - v;
}

// comp layout per cloud (float, n_pad = n rounded up to 4, inside a block sized for n rounded up to 128):
// x[n_pad] y[n_pad] z[n_pad] oidx[n_pad]
template <bool FITS_REG>
__global__ void __launch_bounds__(TPB, 1) fps_flat_kernel(const float* __restrict__ xyz_all, int n, int m,
                                                     int* __restrict__ idx_all, float* __restrict__ out_all,
                                                     float* __restrict__ comp_all, float* __restrict__ temp_all) {
  extern __shared__ __align__(16) float sm[];
  float* const sx = sm;
  float* const sy = sm + SMEM_CAP;
  float* const sz = sm + 2 * SMEM_CAP;
  __shared__ int wsum[NW];
  __shared__ WinSlot slots[2][NW];

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const long long cloud = blockIdx.x;
  const float* const xyz = xyz_all + cloud * n * 3;
  int* const idx = idx_all + cloud * m;
  const int n_pad = (n + 3) & ~3;
  float* const cx = comp_all + cloud * 4 * n_pad;
  float* const cy = cx + n_pad;
  float* const cz = cy + n_pad;
  int* const co = reinterpret_cast<int*>(cz + n_pad);

  // ---- prologue: compaction in the reference's tie-break order ----
  int L = 0;
  while ((2 << L) <= n && L < 9) ++L;      // T = 2^L = min(2^floor(log2 n), 512)
  const int T = 1 << L;
  const int vt = tid < T ? (int)bitrev((unsigned)tid, L) : 0;   // the reference thread this rank stands for
  int cnt = 0;
  if (tid < T) {
    for (int k = vt; k < n; k += T) {
      const float x = xyz[3 * k], y = xyz[3 * k + 1], z = xyz[3 * k + 2];
      const float mag = fmaf(z, z, fmaf(x, x, y * y));
      cnt += !((double)mag <= 1e-3);
    }
  }
  int E;
  int off = block_exscan(cnt, &E, wsum);
  if (tid < T) {
    for (int k = vt; k < n; k += T) {
      const float x = xyz[3 * k], y = xyz[3 * k + 1], z = xyz[3 * k + 2];
      const float mag = fmaf(z, z, fmaf(x, x, y * y));
      if (!((double)mag <= 1e-3)) {
        cx[off] = x; cy[off] = y; cz[off] = z; co[off] = k;
        if (off < SMEM_CAP) { sx[off] = x; sy[off] = y; sz[off] = z; }
        ++off;
      }
    }
  }
  // pad the compact copy to a multiple of 4 so that whole groups can be loaded
  const int E_pad = (E + 3) & ~3;
  if (tid < E_pad - E) {
    const int e = E + tid;
    cx[e] = 0.f; cy[e] = 0.f; cz[e] = 0.f; co[e] = 0;
    if (e < SMEM_CAP) { sx[e] = 0.f; sy[e] = 0.f; sz[e] = 0.f; }
  }
  __threadfence_block();
  __syncthreads();

  if (tid == 0) idx[0] = 0;
  if (E == 0) {                          // nothing eligible: the reference returns index 0 throughout
    for (int j = 1 + tid; j < m; j += TPB) idx[j] = 0;
  } else {
    const int ngroups = (E_pad / 4 + TPB - 1) / TPB;      // groups per thread actually in use
    float temp[FITS_REG ? GROUPS_MAX : 1][4];
    float* const tg = FITS_REG ? nullptr : temp_all + cloud * n_pad;   // spill path for n > REG_CAP
    if (FITS_REG) {
      #pragma unroll
      for (int i = 0; i < GROUPS_MAX; ++i) {
        const int e0 = 4 * (i * TPB + tid);
        #pragma unroll
        for (int q = 0; q < 4; ++q) temp[i][q] = (e0 + q < E) ? 1e10f : -1.0f;
      }
    } else {
      for (int e = tid; e < E_pad; e += TPB) tg[e] = e < E ? 1e10f : -1.0f;
      __syncthreads();
    }

    float ccx = xyz[0], ccy = xyz[1], ccz = xyz[2];       // centre of the first iteration: point 0 as given
    for (int j = 1; j < m; ++j) {
      const f32x2 c2x = pack2(ccx, ccx), c2y = pack2(ccy, ccy), c2z = pack2(ccz, ccz);
      float best = -1.0f;
      int be = 0;

      auto visit = [&](int i, float (&tq)[4]) {
        const int g = i * TPB + tid;            // group index; points 4g..4g+3
        const int e0 = 4 * g;
        float4 px, py, pz;
        if (e0 < SMEM_CAP) {
          px = *reinterpret_cast<const float4*>(sx + e0);
          py = *reinterpret_cast<const float4*>(sy + e0);
          pz = *reinterpret_cast<const float4*>(sz + e0);
        } else {
          px = *reinterpret_cast<const float4*>(cx + e0);
          py = *reinterpret_cast<const float4*>(cy + e0);
          pz = *reinterpret_cast<const float4*>(cz + e0);
        }
        const f32x2 dx0 = sub2(pack2(px.x, px.y), c2x), dx1 = sub2(pack2(px.z, px.w), c2x);
        const f32x2 dy0 = sub2(pack2(py.x, py.y), c2y), dy1 = sub2(pack2(py.z, py.w), c2y);
        const f32x2 dz0 = sub2(pack2(pz.x, pz.y), c2z), dz1 = sub2(pack2(pz.z, pz.w), c2z);
        const f32x2 d0 = fma2(dz0, dz0, fma2(dx0, dx0, mul2(dy0, dy0)));
        const f32x2 d1 = fma2(dz1, dz1, fma2(dx1, dx1, mul2(dy1, dy1)));
        float d[4];
        unpack2(d0, d[0], d[1]);
        unpack2(d1, d[2], d[3]);
        #pragma unroll
        for (int q = 0; q < 4; ++q) {
          const float t = fminf(d[q], tq[q]);
          tq[q] = t;
          const bool gt = t > best;             // strict: ascending compact index keeps the tie rule
          best = gt ? t : best;
          be = gt ? e0 + q : be;
        }
      };

      if (FITS_REG) {
        #pragma unroll
        for (int i = 0; i < GROUPS_MAX; ++i) {
          if (i < ngroups) visit(i, temp[i]);
        }
      } else {
        for (int i = 0; i < ngroups; ++i) {
          const int e0 = 4 * (i * TPB + tid);
          if (e0 < E_pad) {
            float4 t4 = *reinterpret_cast<float4*>(tg + e0);
            float tq[4] = {t4.x, t4.y, t4.z, t4.w};
            visit(i, tq);
            *reinterpret_cast<float4*>(tg + e0) = make_float4(tq[0], tq[1], tq[2], tq[3]);
          }
        }
      }

      // warp arg-max: value first (non-negative floats order like their bit patterns), then lowest e
      const unsigned vb = best < 0.f ? 0u : __float_as_uint(best);
      const unsigned vmax = __reduce_max_sync(0xffffffffu, vb);
      const unsigned ecand = (vb == vmax && !(best < 0.f)) ? (unsigned)be : 0xffffffffu;
      const unsigned emin = __reduce_min_sync(0xffffffffu, ecand);
      const int par = j & 1;
      if (lane == 0) { slots[par][warp].val = vmax; slots[par][warp].e = emin; }
      __syncthreads();
      const WinSlot s = slots[par][lane & (NW - 1)];
      const unsigned V = __reduce_max_sync(0xffffffffu, s.val);
      const unsigned ew = __reduce_min_sync(0xffffffffu, s.val == V ? s.e : 0xffffffffu);
      // ew is always a real point here because E >= 1 (some temp >= 0 exists)
      if (ew < (unsigned)SMEM_CAP) { ccx = sx[ew]; ccy = sy[ew]; ccz = sz[ew]; }
      else { ccx = cx[ew]; ccy = cy[ew]; ccz = cz[ew]; }
      if (tid == 0) idx[j] = (int)ew;          // compact index for now; translated below
    }
    __threadfence_block();
    __syncthreads();
    for (int j = 1 + tid; j < m; j += TPB) idx[j] = co[idx[j]];
  }

  if (out_all != nullptr) {                   // fused gather of the sampled points, (m,3) per cloud
    __threadfence_block();
    __syncthreads();
    float* const out = out_all + cloud * m * 3;
    for (int j = tid; j < m; j += TPB) {
      const int k = idx[j];
      out[3 * j] = xyz[3 * k]; out[3 * j + 1] = xyz[3 * k + 1]; out[3 * j + 2] = xyz[3 * k + 2];
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Pruned kernel
// ------------------------------------------------------------------------------------------------
constexpr int CELLS = 4096;                       // 32 x 32 (Morton) x 4 grid over the eligible points' box
constexpr int BUCKET = 128;                       // points per (warp, slot) = 32 lanes x 4
constexpr int BUCKETS_MAX = NW * GROUPS_MAX;      // 256
constexpr int PR_CAP = 17792;                     // points with smem-resident coordinates (139 buckets)
constexpr int PR_REGION_A = 16384;                // cell counters in the prologue, then boxes + records + winner list
constexpr int PR_ELIST = 1536;                    // winners kept in smem (compact positions); more samples spill to idx[]
constexpr int PR_SMEM_BYTES = PR_CAP * 12 + PR_REGION_A;

struct BucketRec { float maxT; int e; };            // best point of a bucket: its distance and compact position
struct WinRec { unsigned val; int e; };

__device__ __forceinline__ unsigned spread5(unsigned v) {        // abcde -> a0b0c0d0e (Morton spread)
  v = (v | (v << 4)) & 0x0f0f0f0fu;
  v = (v | (v << 2)) & 0x33333333u;
  v = (v | (v << 1)) & 0x55555555u;
  return v;
}

__device__ __forceinline__ float warp_min_f(float v) {
  #pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fminf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ float warp_max_f(float v) {
  #pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// comp layout per cloud (n128 = n rounded up to 128): x[n128] y[n128] z[n128] oidx[n128]
__global__ void __launch_bounds__(TPB, 1) fps_pruned_kernel(const float* __restrict__ xyz_all, int n, int m,
                                                            int* __restrict__ idx_all, float* __restrict__ out_all,
                                                            float* __restrict__ comp_all) {
  extern __shared__ __align__(16) unsigned char smraw[];
  float* const sx = reinterpret_cast<float*>(smraw);
  float* const sy = sx + PR_CAP;
  float* const sz = sy + PR_CAP;
  unsigned char* const regionA = smraw + PR_CAP * 12;
  int* const cells = reinterpret_cast<int*>(regionA);
  float4* const blo = reinterpret_cast<float4*>(regionA);
  float4* const bhi = blo + BUCKETS_MAX;
  BucketRec* const rec = reinterpret_cast<BucketRec*>(bhi + BUCKETS_MAX);      // 8 KB + 2 KB
  int* const elist = reinterpret_cast<int*>(rec + BUCKETS_MAX);                // 6 KB: 16 KB in all
  __shared__ float red[NW][8];
  __shared__ int wsum[NW];
  __shared__ WinRec slots[2][NW];
  __shared__ uint64_t stage_bar;

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const long long cloud = blockIdx.x;
  const float* const xyz = xyz_all + cloud * n * 3;
  int* const idx = idx_all + cloud * m;
  const int n128 = (n + BUCKET - 1) / BUCKET * BUCKET;
  float* const cx = comp_all + cloud * 4 * n128;
  float* const cy = cx + n128;
  float* const cz = cy + n128;
  int* const co = reinterpret_cast<int*>(cz + n128);
  const float inf = __int_as_float(0x7f800000);
  if (tid == 0) { mbar_init(&stage_bar, 1); mbar_fence_init(); }

  // tie key of the reference: (bitreverse_L(k mod T), k div T) as one integer
  int L = 0;
  while ((2 << L) <= n && L < 9) ++L;
  const unsigned T = 1u << L, nq = (unsigned)((n + (int)T - 1) >> L);
  auto tiekey = [&](int k) -> unsigned { return bitrev((unsigned)k & (T - 1), L) * nq + ((unsigned)k >> L); };

  // ---- pass 1: eligibility, count, bounding box ----
  int cnt = 0;
  float lo[3] = {inf, inf, inf}, hi[3] = {-inf, -inf, -inf};
  for (int k = tid; k < n; k += TPB) {
    const float x = xyz[3 * k], y = xyz[3 * k + 1], z = xyz[3 * k + 2];
    const float mag = fmaf(z, z, fmaf(x, x, y * y));
    if (!((double)mag <= 1e-3)) {
      ++cnt;
      lo[0] = fminf(lo[0], x); lo[1] = fminf(lo[1], y); lo[2] = fminf(lo[2], z);
      hi[0] = fmaxf(hi[0], x); hi[1] = fmaxf(hi[1], y); hi[2] = fmaxf(hi[2], z);
    }
  }
  #pragma unroll
  for (int a = 0; a < 3; ++a) { lo[a] = warp_min_f(lo[a]); hi[a] = warp_max_f(hi[a]); }
  cnt = __reduce_add_sync(0xffffffffu, cnt);
  if (lane == 0) {
    red[warp][0] = lo[0]; red[warp][1] = lo[1]; red[warp][2] = lo[2];
    red[warp][3] = hi[0]; red[warp][4] = hi[1]; red[warp][5] = hi[2];
    wsum[warp] = cnt;
  }
  for (int c = tid; c < CELLS; c += TPB) cells[c] = 0;
  __syncthreads();
  int E = 0;
  #pragma unroll
  for (int w = 0; w < NW; ++w) {
    E += wsum[w];
    #pragma unroll
    for (int a = 0; a < 3; ++a) { lo[a] = fminf(lo[a], red[w][a]); hi[a] = fmaxf(hi[a], red[w][3 + a]); }
  }

  if (tid == 0) idx[0] = 0;
  if (E == 0) {                          // nothing eligible: the reference returns index 0 throughout
    for (int j = 1 + tid; j < m; j += TPB) idx[j] = 0;
  } else {
    // ---- pass 2/3: counting sort by grid cell (order inside a cell is irrelevant for the result) ----
    const float sxs = hi[0] > lo[0] ? 32.0f / (hi[0] - lo[0]) : 0.0f;
    const float sys = hi[1] > lo[1] ? 32.0f / (hi[1] - lo[1]) : 0.0f;
    const float szs = hi[2] > lo[2] ? 4.0f / (hi[2] - lo[2]) : 0.0f;
    auto cell_of = [&](float x, float y, float z) -> int {
      const int ix = min(31, max(0, (int)((x - lo[0]) * sxs)));
      const int iy = min(31, max(0, (int)((y - lo[1]) * sys)));
      const int iz = min(3, max(0, (int)((z - lo[2]) * szs)));
      return (int)(((spread5((unsigned)ix) | (spread5((unsigned)iy) << 1)) << 2) | (unsigned)iz);
    };
    for (int k = tid; k < n; k += TPB) {
      const float x = xyz[3 * k], y = xyz[3 * k + 1], z = xyz[3 * k + 2];
      const float mag = fmaf(z, z, fmaf(x, x, y * y));
      if (!((double)mag <= 1e-3)) atomicAdd(&cells[cell_of(x, y, z)], 1);
    }
    __syncthreads();
    {
      constexpr int PER = CELLS / TPB;     // 8 consecutive cells per thread
      int loc[PER], sum = 0;
      #pragma unroll
      for (int c = 0; c < PER; ++c) { loc[c] = cells[tid * PER + c]; sum += loc[c]; }
      int total;
      int base = block_exscan(sum, &total, wsum);
      #pragma unroll
      for (int c = 0; c < PER; ++c) { cells[tid * PER + c] = base; base += loc[c]; }
    }
    __syncthreads();
    for (int k = tid; k < n; k += TPB) {
      const float x = xyz[3 * k], y = xyz[3 * k + 1], z = xyz[3 * k + 2];
      const float mag = fmaf(z, z, fmaf(x, x, y * y));
      if (!((double)mag <= 1e-3)) {
        const int e = atomicAdd(&cells[cell_of(x, y, z)], 1);
        cx[e] = x; cy[e] = y; cz[e] = z; co[e] = k;
      }
    }
    const int E_pad = (E + BUCKET - 1) / BUCKET * BUCKET;
    if (tid < E_pad - E) {               // fill the last bucket; padding never wins (distance -1) nor widens a box
      const int e = E + tid;
      cx[e] = 0.f; cy[e] = 0.f; cz[e] = 0.f; co[e] = 0;
    }
    // The sorted cloud is staged into shared memory by three 1-D TMA bulk copies (UBLKCP) from the
    // L2-resident workspace: make the generic-proxy writes above visible to the async proxy first.
    __threadfence_block();
    asm volatile("fence.proxy.async;" ::: "memory");
    __syncthreads();                     // cell counters are dead from here on: region A becomes boxes + records
    if (tid == 0) {
      const uint32_t bytes = (uint32_t)min(E_pad, PR_CAP) * 4u;
      mbar_expect_tx(&stage_bar, 3u * bytes);
      bulk_g2s(sx, cx, bytes, &stage_bar);
      bulk_g2s(sy, cy, bytes, &stage_bar);
      bulk_g2s(sz, cz, bytes, &stage_bar);
    }
    mbar_wait(&stage_bar, 0u);

    const int nb = E_pad / BUCKET;       // buckets in use; bucket b = slot * NW + warp

    auto load_group = [&](int e0, float4& px, float4& py, float4& pz) {
      if (e0 < PR_CAP) {
        px = *reinterpret_cast<const float4*>(sx + e0);
        py = *reinterpret_cast<const float4*>(sy + e0);
        pz = *reinterpret_cast<const float4*>(sz + e0);
      } else {
        px = *reinterpret_cast<const float4*>(cx + e0);
        py = *reinterpret_cast<const float4*>(cy + e0);
        pz = *reinterpret_cast<const float4*>(cz + e0);
      }
    };

    // ---- bucket boxes, initial records, register-resident distances ----
    float temp[GROUPS_MAX][4];
    #pragma unroll
    for (int i = 0; i < GROUPS_MAX; ++i) {
      const int b = i * NW + warp;
      const int e0 = 4 * (i * TPB + tid);
      #pragma unroll
      for (int q = 0; q < 4; ++q) temp[i][q] = (e0 + q < E) ? 1e10f : -1.0f;
      if (b < nb) {                      // warp-uniform
        float4 px, py, pz;
        load_group(e0, px, py, pz);
        const float X[4] = {px.x, px.y, px.z, px.w}, Y[4] = {py.x, py.y, py.z, py.w}, Z[4] = {pz.x, pz.y, pz.z, pz.w};
        float l0 = inf, l1 = inf, l2 = inf, h0 = -inf, h1 = -inf, h2 = -inf;
        #pragma unroll
        for (int q = 0; q < 4; ++q) {
          if (e0 + q < E) {
            l0 = fminf(l0, X[q]); l1 = fminf(l1, Y[q]); l2 = fminf(l2, Z[q]);
            h0 = fmaxf(h0, X[q]); h1 = fmaxf(h1, Y[q]); h2 = fmaxf(h2, Z[q]);
          }
        }
        l0 = warp_min_f(l0); l1 = warp_min_f(l1); l2 = warp_min_f(l2);
        h0 = warp_max_f(h0); h1 = warp_max_f(h1); h2 = warp_max_f(h2);
        if (lane == 0) {
          // records of one warp are contiguous (slot-major per warp): the per-lane reads below are conflict-free
          const int sidx = warp * GROUPS_MAX + i;
          blo[sidx] = make_float4(l0, l1, l2, 0.f); bhi[sidx] = make_float4(h0, h1, h2, 0.f);
          rec[sidx] = BucketRec{1e10f, e0};   // every bucket is touched in iteration 1 (LB < 1e10) before this is read
        }
      }
    }
    __syncthreads();

    float ccx = xyz[0], ccy = xyz[1], ccz = xyz[2];       // centre of the first iteration: point 0 as given
    for (int j = 1; j < m; ++j) {
      // (a) one bucket per lane: can the new centre lower any distance in it?
      const int btest = lane * NW + warp;                       // slot `lane` of this warp
      const bool bvalid = lane < GROUPS_MAX && btest < nb;
      const int bsafe = warp * GROUPS_MAX + (bvalid ? lane : 0);   // storage index of that bucket's box/record
      bool upd;
      {
        const float4 l4 = blo[bsafe], h4 = bhi[bsafe];
        const float mt = rec[bsafe].maxT;
        const float gx = max3(0.0f, l4.x - ccx, ccx - h4.x);
        const float gy = max3(0.0f, l4.y - ccy, ccy - h4.y);
        const float gz = max3(0.0f, l4.z - ccz, ccz - h4.z);
        const float lb = fmaf(gz, gz, fmaf(gx, gx, __fmul_rn(gy, gy)));   // <= d(k) for every k in the box
        upd = bvalid && lb < mt;
      }
      const unsigned need = __ballot_sync(0xffffffffu, upd);
      __syncwarp();      // orders the record reads above before the record writes below (other lanes)

      // (b) update the buckets that may change and re-elect their best point. Distances live in
      //     registers, so the slot is selected through a jump table instead of 16 predicated blocks.
      const f32x2 c2x = pack2(ccx, ccx), c2y = pack2(ccy, ccy), c2z = pack2(ccz, ccz);
      auto update = [&](int i, float (&tq)[4]) {
        const int e0 = 4 * (i * TPB + tid);
        float4 px, py, pz;
        load_group(e0, px, py, pz);
        const f32x2 dx0 = sub2(pack2(px.x, px.y), c2x), dx1 = sub2(pack2(px.z, px.w), c2x);
        const f32x2 dy0 = sub2(pack2(py.x, py.y), c2y), dy1 = sub2(pack2(py.z, py.w), c2y);
        const f32x2 dz0 = sub2(pack2(pz.x, pz.y), c2z), dz1 = sub2(pack2(pz.z, pz.w), c2z);
        const f32x2 d0 = fma2(dz0, dz0, fma2(dx0, dx0, mul2(dy0, dy0)));
        const f32x2 d1 = fma2(dz1, dz1, fma2(dx1, dx1, mul2(dy1, dy1)));
        float d[4];
        unpack2(d0, d[0], d[1]);
        unpack2(d1, d[2], d[3]);
        #pragma unroll
        for (int q = 0; q < 4; ++q) tq[q] = fminf(d[q], tq[q]);
        const float m4 = fmaxf(fmaxf(tq[0], tq[1]), fmaxf(tq[2], tq[3]));
        const unsigned vb = m4 < 0.f ? 0u : __float_as_uint(m4);          // padding (-1) never competes
        const unsigned vmax = __reduce_max_sync(0xffffffffu, vb);
        // candidates: real points whose distance equals the bucket maximum
        unsigned cm = 0u;
        #pragma unroll
        for (int q = 0; q < 4; ++q) cm |= (e0 + q < E && __float_as_uint(tq[q]) == vmax) ? (1u << q) : 0u;
        const unsigned lanes = __ballot_sync(0xffffffffu, cm != 0u);
        const unsigned multi = __ballot_sync(0xffffffffu, (cm & (cm - 1)) != 0u);
        int ebest = e0 + __ffs(cm) - 1;
        if ((lanes & (lanes - 1)) != 0u || multi != 0u) {                 // warp-uniform; rare: exact tie -> the reference's key decides
          unsigned lk = 0xffffffffu;
          #pragma unroll
          for (int q = 0; q < 4; ++q) {
            if (cm & (1u << q)) {
              const unsigned key = tiekey(co[e0 + q]);
              if (key < lk) { lk = key; ebest = e0 + q; }
            }
          }
          const unsigned kmin = __reduce_min_sync(0xffffffffu, lk);
          if (lk == kmin && cm != 0u) rec[warp * GROUPS_MAX + i] = BucketRec{__uint_as_float(vmax), ebest};
        } else if (cm != 0u) {
          rec[warp * GROUPS_MAX + i] = BucketRec{__uint_as_float(vmax), ebest};
        }
      };
      for (unsigned todo = need; todo != 0u; todo &= todo - 1u) {          // warp-uniform
        switch (__ffs(todo) - 1) {
          case 0: update(0, temp[0]); break;    case 1: update(1, temp[1]); break;
          case 2: update(2, temp[2]); break;    case 3: update(3, temp[3]); break;
          case 4: update(4, temp[4]); break;    case 5: update(5, temp[5]); break;
          case 6: update(6, temp[6]); break;    case 7: update(7, temp[7]); break;
          case 8: update(8, temp[8]); break;    case 9: update(9, temp[9]); break;
          case 10: update(10, temp[10]); break; case 11: update(11, temp[11]); break;
          case 12: update(12, temp[12]); break; case 13: update(13, temp[13]); break;
          case 14: update(14, temp[14]); break; default: update(15, temp[15]); break;
        }
      }
      __syncwarp();

      // (c) best bucket of this warp, (d) best warp of the block; ties go through the key (rare)
      const BucketRec rr = rec[bsafe];
      const unsigned vb = bvalid ? __float_as_uint(rr.maxT) : 0u;           // maxT >= 0 for every bucket in use
      int e = bvalid ? rr.e : -1;
      const unsigned V = __reduce_max_sync(0xffffffffu, vb);
      unsigned cand = __ballot_sync(0xffffffffu, e >= 0 && vb == V);
      if ((cand & (cand - 1)) != 0u) {
        const unsigned key = (e >= 0 && vb == V) ? tiekey(co[e]) : 0xffffffffu;
        const unsigned kmin = __reduce_min_sync(0xffffffffu, key);
        cand = __ballot_sync(0xffffffffu, key == kmin);
      }
      e = __shfl_sync(0xffffffffu, e, __ffs(cand) - 1);
      const int par = j & 1;
      if (lane == 0) slots[par][warp] = WinRec{cand ? V : 0u, cand ? e : -1};
      __syncthreads();
      const WinRec s2 = slots[par][lane & (NW - 1)];
      const unsigned VV = __reduce_max_sync(0xffffffffu, s2.val);
      unsigned cand2 = __ballot_sync(0xffffffffu, lane < NW && s2.e >= 0 && s2.val == VV);
      if ((cand2 & (cand2 - 1)) != 0u) {
        const unsigned key = (lane < NW && s2.e >= 0 && s2.val == VV) ? tiekey(co[s2.e]) : 0xffffffffu;
        const unsigned kmin = __reduce_min_sync(0xffffffffu, key);
        cand2 = __ballot_sync(0xffffffffu, key == kmin);
      }
      const int ew = __shfl_sync(0xffffffffu, s2.e, __ffs(cand2) - 1);
      if (ew < PR_CAP) { ccx = sx[ew]; ccy = sy[ew]; ccz = sz[ew]; }
      else { ccx = cx[ew]; ccy = cy[ew]; ccz = cz[ew]; }
      if (tid == 0) { if (j < PR_ELIST) elist[j] = ew; else idx[j] = ew; }   // compact position; translated below
    }
    __threadfence_block();
    __syncthreads();
    for (int j = 1 + tid; j < m; j += TPB) idx[j] = co[j < PR_ELIST ? elist[j] : idx[j]];
  }

  if (out_all != nullptr) {                   // fused gather of the sampled points, (m,3) per cloud
    __threadfence_block();
    __syncthreads();
    float* const out = out_all + cloud * m * 3;
    for (int j = tid; j < m; j += TPB) {
      const int k = idx[j];
      out[3 * j] = xyz[3 * k]; out[3 * j + 1] = xyz[3 * k + 1]; out[3 * j + 2] = xyz[3 * k + 2];
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Pruned kernel, throughput variant: same algorithm, but nothing large is on chip. Coordinates and
// running distances stay in the L2-resident workspace (a pruned iteration touches ~6 % of them),
// only the bucket boxes/records live in shared memory, so up to six clouds share one SM and overlap
// each other's per-iteration latency chain (prune test -> update -> REDUX -> barrier -> REDUX).
// Records carry the winner's coordinates so the next centre never costs an L2 round trip.
// ------------------------------------------------------------------------------------------------
constexpr int MT_TPB = 256;
constexpr int MT_NW = MT_TPB / 32;                 // 8 warps; lane l of a warp tests the warp's slot l
constexpr int MT_BUCKETS = MT_NW * 32;             // 256 buckets = 32768 points
constexpr int MT_ELIST = 1536;
constexpr int MT_SMEM_BYTES = MT_BUCKETS * (16 + 16 + 32 + 4) + MT_ELIST * 4;   // boxes + records + max distances + winner list = 23 KB
static_assert(MT_SMEM_BYTES >= CELLS * 4, "the cell counters alias the box/record region");

struct MtRec { float maxT; int e; float x, y, z; float pad0, pad1, pad2; };   // 32 B
struct MtWin { unsigned val; int e; float x, y, z; };
// CHIP variant: the running distances of the first MT_DCAP eligible points live in shared memory (56 KB), three
// clouds per SM. Only the read-only coordinates of a touched bucket then travel from L2, and the clouds in flight
// (444 x 15.6 k points x 12 B = 83 MB) fit the 126 MB L2: the six-clouds-per-SM layout keeps 277 MB of coordinates,
// distances and indices in flight and pays 13 GB of DRAM traffic per 888 clouds for it (profiles/SUMMARY_r1.md).
constexpr int MT_DCAP = 14336;                   // 56 KB of distances + 17 KB of boxes/records: three clouds per SM
constexpr int MT_CHIP_SMEM_BYTES = MT_SMEM_BYTES - MT_ELIST * 4 + MT_DCAP * 4;      // no winner list: picks go straight to idx[]

// comp layout per cloud: x[n128] y[n128] z[n128] oidx[n128]; dist_all: t[n128]
template <bool CHIP>
__global__ void __launch_bounds__(MT_TPB, CHIP ? 3 : 6) fps_multi_kernel(const float* __restrict__ xyz_all, int n, int m,
                                                              int* __restrict__ idx_all, float* __restrict__ out_all,
                                                              float* __restrict__ comp_all, float* __restrict__ dist_all) {
  extern __shared__ __align__(16) unsigned char smraw[];
  float* const sdist = reinterpret_cast<float*>(smraw + MT_SMEM_BYTES - MT_ELIST * 4);      // CHIP only: distances of points [0, MT_DCAP), in place of the winner list
  int* const cells = reinterpret_cast<int*>(smraw);
  float4* const blo = reinterpret_cast<float4*>(smraw);
  float4* const bhi = blo + MT_BUCKETS;
  MtRec* const rec = reinterpret_cast<MtRec*>(bhi + MT_BUCKETS);
  float* const bmax = reinterpret_cast<float*>(rec + MT_BUCKETS);   // rec[].maxT again, densely: the per-lane compare key
  int* const elist = reinterpret_cast<int*>(bmax + MT_BUCKETS);
  __shared__ float red[MT_NW][8];
  __shared__ int wsum[MT_NW];
  __shared__ MtWin slots[2][MT_NW];

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const long long cloud = blockIdx.x;
  const float* const xyz = xyz_all + cloud * n * 3;
  int* const idx = idx_all + cloud * m;
  const int n128 = (n + BUCKET - 1) / BUCKET * BUCKET;
  // Bucket-major workspace: bucket k holds x[128] y[128] z[128] t[128] o[128] (2560 contiguous bytes), so one
  // address plus immediates serves the four 128-bit loads and the store of an update (the planar layout
  // cost ~20 instructions of 64-bit pointer arithmetic per touched bucket at this kernel's 40 registers).
  // The comp (4 n128) and temp (n128) regions of the workspace are contiguous: 5 n128 floats per cloud.
  (void)dist_all;
  float* const cb = comp_all + cloud * 5 * n128;
  auto at = [&](int e, int comp) -> float* { return cb + (e >> 7) * (5 * BUCKET) + comp * BUCKET + (e & (BUCKET - 1)); };
  auto orig = [&](int e) -> int { return *reinterpret_cast<const int*>(at(e, 4)); };
  const float inf = __int_as_float(0x7f800000);

  int L = 0;
  while ((2 << L) <= n && L < 9) ++L;
  const unsigned T = 1u << L, nq = (unsigned)((n + (int)T - 1) >> L);
  auto tiekey = [&](int k) -> unsigned { return bitrev((unsigned)k & (T - 1), L) * nq + ((unsigned)k >> L); };

  // ---- pass 1: eligibility, count, bounding box ----
  int cnt = 0;
  float lo[3] = {inf, inf, inf}, hi[3] = {-inf, -inf, -inf};
  for (int k = tid; k < n; k += MT_TPB) {
    const float x = xyz[3 * k], y = xyz[3 * k + 1], z = xyz[3 * k + 2];
    const float mag = fmaf(z, z, fmaf(x, x, y * y));
    if (!((double)mag <= 1e-3)) {
      ++cnt;
      lo[0] = fminf(lo[0], x); lo[1] = fminf(lo[1], y); lo[2] = fminf(lo[2], z);
      hi[0] = fmaxf(hi[0], x); hi[1] = fmaxf(hi[1], y); hi[2] = fmaxf(hi[2], z);
    }
  }
  #pragma unroll
  for (int a = 0; a < 3; ++a) { lo[a] = warp_min_f(lo[a]); hi[a] = warp_max_f(hi[a]); }
  cnt = __reduce_add_sync(0xffffffffu, cnt);
  if (lane == 0) {
    red[warp][0] = lo[0]; red[warp][1] = lo[1]; red[warp][2] = lo[2];
    red[warp][3] = hi[0]; red[warp][4] = hi[1]; red[warp][5] = hi[2];
    wsum[warp] = cnt;
  }
  for (int c = tid; c < CELLS; c += MT_TPB) cells[c] = 0;
  __syncthreads();
  int E = 0;
  #pragma unroll
  for (int w = 0; w < MT_NW; ++w) {
    E += wsum[w];
    #pragma unroll
    for (int a = 0; a < 3; ++a) { lo[a] = fminf(lo[a], red[w][a]); hi[a] = fmaxf(hi[a], red[w][3 + a]); }
  }
  __syncthreads();

  if (tid == 0) idx[0] = 0;
  if (E == 0) {
    for (int j = 1 + tid; j < m; j += MT_TPB) idx[j] = 0;
  } else {
    // ---- counting sort by grid cell into the workspace ----
    const float sxs = hi[0] > lo[0] ? 32.0f / (hi[0] - lo[0]) : 0.0f;
    const float sys = hi[1] > lo[1] ? 32.0f / (hi[1] - lo[1]) : 0.0f;
    const float szs = hi[2] > lo[2] ? 4.0f / (hi[2] - lo[2]) : 0.0f;
    auto cell_of = [&](float x, float y, float z) -> int {
      const int ix = min(31, max(0, (int)((x - lo[0]) * sxs)));
      const int iy = min(31, max(0, (int)((y - lo[1]) * sys)));
      const int iz = min(3, max(0, (int)((z - lo[2]) * szs)));
      return (int)(((spread5((unsigned)ix) | (spread5((unsigned)iy) << 1)) << 2) | (unsigned)iz);
    };
    for (int k = tid; k < n; k += MT_TPB) {
      const float x = xyz[3 * k], y = xyz[3 * k + 1], z = xyz[3 * k + 2];
      const float mag = fmaf(z, z, fmaf(x, x, y * y));
      if (!((double)mag <= 1e-3)) atomicAdd(&cells[cell_of(x, y, z)], 1);
    }
    __syncthreads();
    {
      constexpr int PER = CELLS / MT_TPB;     // 16 consecutive cells per thread
      int sum = 0;
      #pragma unroll
      for (int c = 0; c < PER; ++c) sum += cells[tid * PER + c];
      // block exclusive scan over 256 threads
      int inc = sum;
      #pragma unroll
      for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += t; }
      if (lane == 31) wsum[warp] = inc;
      __syncthreads();
      int base = inc - sum;
      #pragma unroll
      for (int w = 0; w < MT_NW; ++w) if (w < warp) base += wsum[w];
      #pragma unroll
      for (int c = 0; c < PER; ++c) { const int v = cells[tid * PER + c]; cells[tid * PER + c] = base; base += v; }
    }
    __syncthreads();
    for (int k = tid; k < n; k += MT_TPB) {
      const float x = xyz[3 * k], y = xyz[3 * k + 1], z = xyz[3 * k + 2];
      const float mag = fmaf(z, z, fmaf(x, x, y * y));
      if (!((double)mag <= 1e-3)) {
        const int e = atomicAdd(&cells[cell_of(x, y, z)], 1);
        *at(e, 0) = x; *at(e, 1) = y; *at(e, 2) = z; *reinterpret_cast<int*>(at(e, 4)) = k;
        if (CHIP && e < MT_DCAP) sdist[e] = 1e10f; else *at(e, 3) = 1e10f;
      }
    }
    const int E_pad = (E + BUCKET - 1) / BUCKET * BUCKET;
    if (tid < E_pad - E) {
      const int e = E + tid;
      *at(e, 0) = 0.f; *at(e, 1) = 0.f; *at(e, 2) = 0.f; *reinterpret_cast<int*>(at(e, 4)) = 0;
      if (CHIP && e < MT_DCAP) sdist[e] = -1.0f; else *at(e, 3) = -1.0f;
    }
    __threadfence_block();
    __syncthreads();                     // cell counters are dead: the region becomes boxes + records

    const int nb = E_pad / BUCKET;       // bucket b = slot * MT_NW + warp; points [128 b, 128 b + 128)

    for (int b = warp; b < nb; b += MT_NW) {
      const int e0 = b * BUCKET + 4 * lane;
      const float* const pb = cb + b * (5 * BUCKET) + 4 * lane;
      const float4 px = *reinterpret_cast<const float4*>(pb);
      const float4 py = *reinterpret_cast<const float4*>(pb + BUCKET);
      const float4 pz = *reinterpret_cast<const float4*>(pb + 2 * BUCKET);
      const float X[4] = {px.x, px.y, px.z, px.w}, Y[4] = {py.x, py.y, py.z, py.w}, Z[4] = {pz.x, pz.y, pz.z, pz.w};
      float l0 = inf, l1 = inf, l2 = inf, h0 = -inf, h1 = -inf, h2 = -inf;
      #pragma unroll
      for (int q = 0; q < 4; ++q) {
        if (e0 + q < E) {
          l0 = fminf(l0, X[q]); l1 = fminf(l1, Y[q]); l2 = fminf(l2, Z[q]);
          h0 = fmaxf(h0, X[q]); h1 = fmaxf(h1, Y[q]); h2 = fmaxf(h2, Z[q]);
        }
      }
      l0 = warp_min_f(l0); l1 = warp_min_f(l1); l2 = warp_min_f(l2);
      h0 = warp_max_f(h0); h1 = warp_max_f(h1); h2 = warp_max_f(h2);
      if (lane == 0) {
        const int sidx = warp * 32 + b / MT_NW;      // records of one warp are contiguous: conflict-free per-lane reads
        blo[sidx] = make_float4(l0, l1, l2, 0.f); bhi[sidx] = make_float4(h0, h1, h2, 0.f);
        rec[sidx] = MtRec{1e10f, e0, X[0], Y[0], Z[0], 0.f, 0.f, 0.f};   // replaced in iteration 1 (LB < 1e10 everywhere)
        bmax[sidx] = 1e10f;
      }
    }
    __syncthreads();

    float ccx = xyz[0], ccy = xyz[1], ccz = xyz[2];
    for (int j = 1; j < m; ++j) {
      // (a) lane l tests the warp's slot l
      const int btest = lane * MT_NW + warp;
      const bool bvalid = btest < nb;
      const int bsafe = warp * 32 + (bvalid ? lane : 0);        // storage index of that bucket's box/record
      bool upd;
      {
        const float4 l4 = blo[bsafe], h4 = bhi[bsafe];
        const float mt = bmax[bsafe];
        const float gx = max3(0.0f, l4.x - ccx, ccx - h4.x);
        const float gy = max3(0.0f, l4.y - ccy, ccy - h4.y);
        const float gz = max3(0.0f, l4.z - ccz, ccz - h4.z);
        const float lb = fmaf(gz, gz, fmaf(gx, gx, __fmul_rn(gy, gy)));
        upd = bvalid && lb < mt;
      }
      const unsigned need = __ballot_sync(0xffffffffu, upd);
      __syncwarp();      // orders the record reads above before the record writes below (other lanes)

      // (b) update the buckets that may change
      const f32x2 c2x = pack2(ccx, ccx), c2y = pack2(ccy, ccy), c2z = pack2(ccz, ccz);
      // The coordinates of a touched bucket come from L2: while one bucket is processed the next one's three
      // 128-bit loads are already in flight (a warp touches 0-3 buckets per iteration).
      float4 nx = make_float4(0, 0, 0, 0), ny = nx, nz = nx;
      if (CHIP && need != 0u) {
        const float* const nb0 = cb + ((__ffs(need) - 1) * MT_NW + warp) * (5 * BUCKET) + 4 * lane;
        nx = *reinterpret_cast<const float4*>(nb0);
        ny = *reinterpret_cast<const float4*>(nb0 + BUCKET);
        nz = *reinterpret_cast<const float4*>(nb0 + 2 * BUCKET);
      }
      for (unsigned todo = need; todo != 0u; todo &= todo - 1u) {
        const int b = (__ffs(todo) - 1) * MT_NW + warp;
        const int e0 = b * BUCKET + 4 * lane;
        float* const pb = cb + b * (5 * BUCKET) + 4 * lane;
        float4 px = nx, py = ny, pz = nz;
        if (!CHIP) {
          px = *reinterpret_cast<const float4*>(pb);
          py = *reinterpret_cast<const float4*>(pb + BUCKET);
          pz = *reinterpret_cast<const float4*>(pb + 2 * BUCKET);
        }
        const unsigned rest = todo & (todo - 1u);
        if (CHIP && rest != 0u) {
          const float* const nb1 = cb + ((__ffs(rest) - 1) * MT_NW + warp) * (5 * BUCKET) + 4 * lane;
          nx = *reinterpret_cast<const float4*>(nb1);
          ny = *reinterpret_cast<const float4*>(nb1 + BUCKET);
          nz = *reinterpret_cast<const float4*>(nb1 + 2 * BUCKET);
        }
        float* const tp = (CHIP && e0 < MT_DCAP) ? sdist + e0 : pb + 3 * BUCKET;        // warp-uniform choice
        const float4 t4 = *reinterpret_cast<const float4*>(tp);
        const f32x2 dx0 = sub2(pack2(px.x, px.y), c2x), dx1 = sub2(pack2(px.z, px.w), c2x);
        const f32x2 dy0 = sub2(pack2(py.x, py.y), c2y), dy1 = sub2(pack2(py.z, py.w), c2y);
        const f32x2 dz0 = sub2(pack2(pz.x, pz.y), c2z), dz1 = sub2(pack2(pz.z, pz.w), c2z);
        const f32x2 d0 = fma2(dz0, dz0, fma2(dx0, dx0, mul2(dy0, dy0)));
        const f32x2 d1 = fma2(dz1, dz1, fma2(dx1, dx1, mul2(dy1, dy1)));
        float d[4];
        unpack2(d0, d[0], d[1]);
        unpack2(d1, d[2], d[3]);
        float tq[4] = {fminf(d[0], t4.x), fminf(d[1], t4.y), fminf(d[2], t4.z), fminf(d[3], t4.w)};
        *reinterpret_cast<float4*>(tp) = make_float4(tq[0], tq[1], tq[2], tq[3]);
        const float m4 = fmaxf(fmaxf(tq[0], tq[1]), fmaxf(tq[2], tq[3]));
        const unsigned vb = m4 < 0.f ? 0u : __float_as_uint(m4);
        const unsigned vmax = __reduce_max_sync(0xffffffffu, vb);
        unsigned cm = 0u;
        #pragma unroll
        for (int q = 0; q < 4; ++q) cm |= (e0 + q < E && __float_as_uint(tq[q]) == vmax) ? (1u << q) : 0u;
        const unsigned lanes = __ballot_sync(0xffffffffu, cm != 0u);
        const unsigned multi = __ballot_sync(0xffffffffu, (cm & (cm - 1)) != 0u);
        int qb = __ffs(cm) - 1;
        bool mine = cm != 0u;
        if ((lanes & (lanes - 1)) != 0u || multi != 0u) {       // warp-uniform; exact tie: the reference's key decides
          unsigned lk = 0xffffffffu;
          #pragma unroll
          for (int q = 0; q < 4; ++q) {
            if (cm & (1u << q)) {
              const unsigned key = tiekey(orig(e0 + q));
              if (key < lk) { lk = key; qb = q; }
            }
          }
          const unsigned kmin = __reduce_min_sync(0xffffffffu, lk);
          mine = cm != 0u && lk == kmin;
        }
        if (mine) {
          const float wx = qb == 0 ? px.x : qb == 1 ? px.y : qb == 2 ? px.z : px.w;
          const float wy = qb == 0 ? py.x : qb == 1 ? py.y : qb == 2 ? py.z : py.w;
          const float wz = qb == 0 ? pz.x : qb == 1 ? pz.y : qb == 2 ? pz.z : pz.w;
          rec[warp * 32 + (__ffs(todo) - 1)] = MtRec{__uint_as_float(vmax), e0 + qb, wx, wy, wz, 0.f, 0.f, 0.f};
          bmax[warp * 32 + (__ffs(todo) - 1)] = __uint_as_float(vmax);
        }
      }
      __syncwarp();

      // (c) best bucket of this warp, (d) best warp of the block
      const unsigned vb = bvalid ? __float_as_uint(bmax[bsafe]) : 0u;
      const unsigned V = __reduce_max_sync(0xffffffffu, vb);
      unsigned cand = __ballot_sync(0xffffffffu, bvalid && vb == V);
      if ((cand & (cand - 1)) != 0u) {
        const unsigned key = (bvalid && vb == V) ? tiekey(orig(rec[bsafe].e)) : 0xffffffffu;
        const unsigned kmin = __reduce_min_sync(0xffffffffu, key);
        cand = __ballot_sync(0xffffffffu, key == kmin);
      }
      const int par = j & 1;
      if (cand == 0u) { if (lane == 0) slots[par][warp] = MtWin{0u, -1, 0.f, 0.f, 0.f}; }
      else if (lane == __ffs(cand) - 1) { const MtRec rr = rec[bsafe]; slots[par][warp] = MtWin{V, rr.e, rr.x, rr.y, rr.z}; }
      __syncthreads();
      const MtWin s2 = slots[par][lane & (MT_NW - 1)];
      const bool sv = lane < MT_NW && s2.e >= 0;
      const unsigned VV = __reduce_max_sync(0xffffffffu, sv ? s2.val : 0u);
      unsigned cand2 = __ballot_sync(0xffffffffu, sv && s2.val == VV);
      if ((cand2 & (cand2 - 1)) != 0u) {
        const unsigned key = (sv && s2.val == VV) ? tiekey(orig(s2.e)) : 0xffffffffu;
        const unsigned kmin = __reduce_min_sync(0xffffffffu, key);
        cand2 = __ballot_sync(0xffffffffu, key == kmin);
      }
      const int src = __ffs(cand2) - 1;
      const int ew = __shfl_sync(0xffffffffu, s2.e, src);
      ccx = __shfl_sync(0xffffffffu, s2.x, src);
      ccy = __shfl_sync(0xffffffffu, s2.y, src);
      ccz = __shfl_sync(0xffffffffu, s2.z, src);
      if (tid == 0) { if (!CHIP && j < MT_ELIST) elist[j] = ew; else idx[j] = ew; }
    }
    __threadfence_block();
    __syncthreads();
    for (int j = 1 + tid; j < m; j += MT_TPB) idx[j] = orig((!CHIP && j < MT_ELIST) ? elist[j] : idx[j]);
  }

  if (out_all != nullptr) {
    __threadfence_block();
    __syncthreads();
    float* const out = out_all + cloud * m * 3;
    for (int j = tid; j < m; j += MT_TPB) {
      const int k = idx[j];
      out[3 * j] = xyz[3 * k]; out[3 * j + 1] = xyz[3 * k + 1]; out[3 * j + 2] = xyz[3 * k + 2];
    }
  }
}

__global__ void __launch_bounds__(256) gather_kernel(const float* __restrict__ points, const int* __restrict__ idx,
                                                     int c, int n, int m, float* __restrict__ out) {
  const int i = blockIdx.z, l = blockIdx.y;
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j < m) out[((long long)i * c + l) * m + j] = points[((long long)i * c + l) * n + idx[(long long)i * m + j]];
}

__global__ void __launch_bounds__(256) gather_grad_kernel(const float* __restrict__ grad_out, const int* __restrict__ idx,
                                                          int c, int n, int m, float* __restrict__ grad_points) {
  const int i = blockIdx.z, l = blockIdx.y;
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j < m)
    atomicAdd(grad_points + ((long long)i * c + l) * n + idx[(long long)i * m + j], grad_out[((long long)i * c + l) * m + j]);
}

}  // namespace fps
}  // namespace dusty

using namespace dusty;
using namespace dusty::fps;

static size_t fps_comp_bytes(int b, int n) { return align_up((size_t)b * 4 * ((n + 127) / 128 * 128) * sizeof(float), 256); }
static size_t fps_temp_bytes(int b, int n) { return align_up((size_t)b * ((n + 127) / 128 * 128) * sizeof(float), 256); }

extern "C" size_t dusty_fps_workspace_bytes(int b, int n, int m) {
  (void)m;
  if (b <= 0 || n <= 0) return 0;
  return fps_comp_bytes(b, n) + fps_temp_bytes(b, n);
}

extern "C" int dusty_fps(const float* xyz, int b, int n, int m, int32_t* idx, float* out_xyz, void* workspace,
                         size_t workspace_bytes, void* stream) {
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (b < 0 || n <= 0 || m < 0) return fail_arg(DUSTY_EINVAL, "fps: bad sizes b=%d n=%d m=%d", b, n, m);
  if (b == 0 || m == 0) return 0;
  if (int rc = check_device()) return rc;
  if (!xyz || !idx || !workspace) return fail_arg(DUSTY_EINVAL, "fps: null pointer");
  if (!aligned16(workspace)) return fail_arg(DUSTY_EALIGN, "fps: workspace must be 16-byte aligned");
  if (workspace_bytes < dusty_fps_workspace_bytes(b, n, m))
    return fail_arg(DUSTY_ENOSPACE, "fps: workspace %zu < %zu", workspace_bytes, dusty_fps_workspace_bytes(b, n, m));
  float* comp = static_cast<float*>(workspace);
  float* temp = reinterpret_cast<float*>(static_cast<char*>(workspace) + fps_comp_bytes(b, n));
  // fps_multi_kernel addresses both regions as one (5 n128 floats per cloud): they must be contiguous
  if (temp != comp + (size_t)b * 4 * ((n + 127) / 128 * 128)) return fail_arg(DUSTY_EINVAL, "fps: workspace regions are not contiguous");
  static bool configured[kMaxDevices] = {};
  static bool force_flat = false, force_single = false, force_multi = false, force_l2 = false;
  const int dev = current_device();
  if (!configured[dev]) {
    DUSTY_CUDA(cudaFuncSetAttribute(fps_flat_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES));
    DUSTY_CUDA(cudaFuncSetAttribute(fps_flat_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES));
    DUSTY_CUDA(cudaFuncSetAttribute(fps_pruned_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, PR_SMEM_BYTES));
    DUSTY_CUDA(cudaFuncSetAttribute(fps_multi_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, MT_SMEM_BYTES));
    DUSTY_CUDA(cudaFuncSetAttribute(fps_multi_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, MT_CHIP_SMEM_BYTES));
    const char* env = getenv("DUSTY_FPS_ALGO");       // A/B switch for profiling: flat | single | multi | l2 (six per SM, distances in L2); same indices from all
    force_flat = env && env[0] == 'f';
    force_single = env && env[0] == 's';
    force_multi = env && env[0] == 'm';
    force_l2 = env && env[0] == 'l';
    configured[dev] = true;
  }
  // more clouds than SMs: four clouds per SM hide each other's latency chain (throughput variant);
  // otherwise one cloud per SM with everything on chip (latency variant)
  const bool multi = force_multi || force_l2 || (!force_single && b > kNumSMs);
  if (n > REG_CAP) fps_flat_kernel<false><<<b, TPB, SMEM_BYTES, st>>>(xyz, n, m, idx, out_xyz, comp, temp);
  else if (force_flat) fps_flat_kernel<true><<<b, TPB, SMEM_BYTES, st>>>(xyz, n, m, idx, out_xyz, comp, temp);
  else if (multi && force_l2) fps_multi_kernel<false><<<b, MT_TPB, MT_SMEM_BYTES, st>>>(xyz, n, m, idx, out_xyz, comp, temp);
  else if (multi) fps_multi_kernel<true><<<b, MT_TPB, MT_CHIP_SMEM_BYTES, st>>>(xyz, n, m, idx, out_xyz, comp, temp);
  else fps_pruned_kernel<<<b, TPB, PR_SMEM_BYTES, st>>>(xyz, n, m, idx, out_xyz, comp);
  DUSTY_AFTER_LAUNCH("fps kernel");
  return 0;
}

extern "C" int dusty_gather_points(const float* points, const int32_t* idx, int b, int c, int n, int m, float* out,
                                   void* stream) {
  if (b < 0 || c < 0 || n <= 0 || m < 0) return fail_arg(DUSTY_EINVAL, "gather_points: bad sizes");
  if (b == 0 || c == 0 || m == 0) return 0;
  if (b > 65535 || c > 65535) return fail_arg(DUSTY_EINVAL, "gather_points: b and c must be <= 65535");
  if (int rc = check_device()) return rc;
  if (!points || !idx || !out) return fail_arg(DUSTY_EINVAL, "gather_points: null pointer");
  gather_kernel<<<dim3((m + 255) / 256, c, b), 256, 0, static_cast<cudaStream_t>(stream)>>>(points, idx, c, n, m, out);
  DUSTY_AFTER_LAUNCH("gather_kernel");
  return 0;
}

extern "C" int dusty_gather_points_grad(const float* grad_out, const int32_t* idx, int b, int c, int n, int m,
                                        float* grad_points, void* stream) {
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (b < 0 || c < 0 || n <= 0 || m < 0) return fail_arg(DUSTY_EINVAL, "gather_points_grad: bad sizes");
  if (b == 0 || c == 0) return 0;
  if (b > 65535 || c > 65535) return fail_arg(DUSTY_EINVAL, "gather_points_grad: b and c must be <= 65535");
  if (int rc = check_device()) return rc;
  if (!grad_points) return fail_arg(DUSTY_EINVAL, "gather_points_grad: null pointer");
  DUSTY_CUDA(cudaMemsetAsync(grad_points, 0, sizeof(float) * (size_t)b * c * n, st));
  if (m == 0) return 0;
  if (!grad_out || !idx) return fail_arg(DUSTY_EINVAL, "gather_points_grad: null pointer");
  gather_grad_kernel<<<dim3((m + 255) / 256, c, b), 256, 0, st>>>(grad_out, idx, c, n, m, grad_points);
  DUSTY_AFTER_LAUNCH("gather_grad_kernel");
  return 0;
}
