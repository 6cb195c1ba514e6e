// Chamfer nearest-neighbour kernels for sm_100a.
//
// Replaces ChamferDistanceKernel (reference utils/metrics/distance/cd/chamfer_distance.cu:6-131),
// its launcher (:133-146) and the Python double loop _pairwise_distance that calls it once per row
// and 512-column block (reference utils/metrics/cov_mmd_1nna.py:24-51).
//
// One kernel, two front ends:
//   * batch  -- dusty_chamfer_forward: per-point (dist, idx) in both directions for b cloud pairs
//   * matrix -- dusty_chamfer_matrix : one CTA per matrix entry (cloud i of A, cloud j of B), both
//               directions, reduced on chip to M[i,j] = mean(dist1) + mean(dist2)  (compute_cd,
//               reference cov_mmd_1nna.py:19-21)
//
// Arithmetic. A directed search keeps R "row" points per thread in registers and streams the
// other cloud through shared memory in 2048-point tiles (1-D TMA bulk copies, double buffered on
// two mbarriers). Tiles are in *scan format*: for points 2q, 2q+1 two float4 {x0,x1,y0,y1}
// {z0,z1,n0,n1} with n = |p|^2, so one LDS.128 pair feeds packed FFMA2 directly.
//   search:  s(a,b) = |b|^2 - 2 a.b  as 3 FFMA2 per two candidates + one 3-input FMNMX, and per
//            32-candidate chunk one compare/select that remembers which chunk holds the minimum;
//   exact :  the winning chunk (1.6 % of the tile) is re-evaluated in the reference's rounding,
//            d = fma(dz,dz,fma(dx,dx,dy*dy)) on differences, and the minimum of those is the
//            result;
//   guard :  the search also keeps the runner-up chunk's minimum. Whenever it lies within
//            delta = 48 u (|a|^2 + D), u = 2^-24, D = the search's own estimate of the distance, of the
//            winner's -- a rigorous bound on (search rounding error of two candidates) + (rounding of the
//            reference formula), derived at search_window() -- the search cannot tell which chunk holds
//            the reference's minimum, and the warp re-evaluates the WHOLE tile for that row in the
//            reference's rounding (32 lanes x 64 candidates, two shuffles). Hence every distance (and
//            index) returned is exactly the reference kernel's, for any finite input; the guard fires for
//            ~0.1 % of the (row, tile) pairs on LiDAR-like clouds and costs < 0.5 %.
#include <algorithm>

#include "common.cuh"

namespace dusty {
namespace chamfer {

constexpr int TPB = 256;
constexpr int TILE = 2048;            // scan points per shared-memory tile (= float4 per tile)
constexpr int CHUNK = 32;             // candidates per search chunk

struct Params {
  const float4* scanX;      // scan-format clouds, X side (rows of the matrix / xyz1)
  const float4* scanY;      // Y side (columns / xyz2)
  long long strideX, strideY;   // float4 per cloud (= padded point count)
  int countX, countY;       // points per cloud
  int paddedX, paddedY;     // counts rounded up to CHUNK
  // matrix front end
  int row_begin, row_stride;
  int symmetric, mirror, compact_rows;
  float* M;
  long long ldm;
  // batch front end
  float* dist1; float* dist2;
  int* idx1; int* idx2;
  // merged-origin clouds: per-cloud {points kept, weight of the last kept point}, the per-chunk bounding boxes of
  // sorted clouds and, for the batch front end, the map from a sorted position back to the original point index
  // (the merged origin point maps to the first zero point)
  const int2* metaX; const int2* metaY;
  const float4* boxX; const float4* boxY;
  const float4* bbX; const float4* bbY;      // boxes of the blocks of 32 chunks (sorted clouds, nn_walk_split_kernel)
  const int* permX; const int* permY;
  unsigned long long* visited;   // measurement only (null: off): (row, candidate) pairs the pruned search really evaluated
  // fused MMD/COV/1-NNA epilogue (matrix front end; null: off). keys = 3 arrays of n_total packed
  // (float bits << 32 | stacked index) minima: [0] leave-one-out nearest neighbour of every stacked cloud,
  // [1] nearest reference cloud of every generated cloud, [2] nearest generated cloud of every reference cloud
  unsigned long long* keys;
  int n_total, n_ref, offX, offY;
};

template <int NT>
__device__ __forceinline__ double block_sum(double v, double* red) {
  #pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  __syncthreads();
  if (lane == 0) red[warp] = v;
  __syncthreads();
  double s = 0.0;
  if (threadIdx.x == 0) {
    #pragma unroll
    for (int w = 0; w < NT / 32; ++w) s += red[w];   // fixed order: result independent of sharding
  }
  return s;
}

// Half-width of the search's blind spot around its own minimum `cur` for a row point a (see the header):
// any candidate the reference kernel could prefer has a search value below cur + window. With u = 2^-24,
// r^2 = D the squared distance of a candidate b, |b| <= |a| + r:
//   search value s~ = fl chain of |b|^2 - 2 a.b: |s~ - s| <= u (6 |b|^2 + 6 |a||b|) <= u (21 |a|^2 + 15 D)
//   reference value d~ = fma(dz,dz,fma(dx,dx,dy*dy)) on rounded differences: |d~ - D| <= 5 u D
// so for the search's winner b^ and the reference's arg-min b* (d~(b*) <= d~(b^) => D(b*) <= (1 + 10u) D(b^)):
//   s~(b*) - s~(b^) <= u (42 |a|^2 + 40 D(b^)),  D(b^) <= (cur + |a|^2)(1 + O(u)).
// 48 u leaves > 12 % for the rounding of this very expression and of the comparison; 1e-36 covers underflow.
__device__ __forceinline__ float search_window(float ax, float ay, float az, float cur) {
  const float an = fmaf(az, az, fmaf(ax, ax, ay * ay));
  return fmaf(2.86102295e-6f /* 48 * 2^-24 */, an + fmaxf(cur + an, 0.0f), 1e-36f);
}

// The whole tile (npairs candidate pairs in scan format) against one row point, in the reference's rounding,
// by all 32 lanes of a warp: minimum and, if wanted, the tile-relative position of the winner -- the lowest
// position among bit-equal minima.
template <bool WANT_INDEX>
__device__ __forceinline__ void warp_tile_exact_min(const float4* tp, int npairs, float ax, float ay, float az, int lane,
                                                    float& best, int& best_pos) {
  const f32x2 ax2 = pack2(ax, ax), ay2 = pack2(ay, ay), az2 = pack2(az, az);
  float e = __int_as_float(0x7f800000);
  int ei = 0x7fffffff;
  for (int q = lane; q < npairs; q += 32) {
    const float4 q0 = tp[2 * q], q1 = tp[2 * q + 1];
    const f32x2 dx = sub2(pack2(q0.x, q0.y), ax2);
    const f32x2 dy = sub2(pack2(q0.z, q0.w), ay2);
    const f32x2 dz = sub2(pack2(q1.x, q1.y), az2);
    float lo, hi;
    unpack2(fma2(dz, dz, fma2(dx, dx, mul2(dy, dy))), lo, hi);
    if (WANT_INDEX) {                       // q ascends: strict < keeps the lane's lowest position
      if (lo < e) { e = lo; ei = 2 * q; }
      if (hi < e) { e = hi; ei = 2 * q + 1; }
    } else {
      e = min3(e, lo, hi);
    }
  }
  float m = e;
  #pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fminf(m, __shfl_xor_sync(0xffffffffu, m, o));
  best = m;
  if (WANT_INDEX) {
    const bool mine = e == m && ei != 0x7fffffff;
    const unsigned key = mine ? (unsigned)ei : 0x7fffffffu;
    const unsigned kmin = __reduce_min_sync(0xffffffffu, key);
    const unsigned who = __ballot_sync(0xffffffffu, mine && key == kmin);
    best_pos = who ? __shfl_sync(0xffffffffu, ei, __ffs(who) - 1) : 0x7fffffff;
  }
}

// DEFERRED guard (merged clouds): one row point against the whole scanned cloud, read from global memory (L2) in the
// reference's rounding by all 32 lanes; a lane takes whole 32-candidate chunks and skips those whose box cannot
// reach `thr`, the exact distance already found in the search's winning chunk (boxes == null: every chunk).
// Returns the minimum and the winner's position (lowest original index among equal minima when perm != null).
template <bool WANT_INDEX>
__device__ __forceinline__ void warp_cloud_exact_min(const float4* cloud, int nchunks, const float4* boxes, float thr,
                                                     float ax, float ay, float az, int lane, const int* perm, float& best,
                                                     int& best_pos) {
  const f32x2 ax2 = pack2(ax, ax), ay2 = pack2(ay, ay), az2 = pack2(az, az);
  float e = __int_as_float(0x7f800000);
  int ei = 0x7fffffff;
  for (int ch = lane; ch < nchunks; ch += 32) {
    if (boxes != nullptr) {
      const float4 bl = boxes[2 * ch], bh = boxes[2 * ch + 1];
      const float gx = max3(0.0f, bl.x - ax, ax - bh.x), gy = max3(0.0f, bl.y - ay, ay - bh.y), gz = max3(0.0f, bl.z - az, az - bh.z);
      if (bl.w == 0.0f && fmaf(gz, gz, fmaf(gx, gx, __fmul_rn(gy, gy))) > thr) continue;      // cannot reach (or tie) thr; .w: holds the origin
    }
    const float4* cp = cloud + (long long)ch * CHUNK;
    #pragma unroll 4
    for (int k = 0; k < CHUNK / 2; ++k) {
      const float4 q0 = cp[2 * k], q1 = cp[2 * k + 1];
      const f32x2 dx = sub2(pack2(q0.x, q0.y), ax2);
      const f32x2 dy = sub2(pack2(q0.z, q0.w), ay2);
      const f32x2 dz = sub2(pack2(q1.x, q1.y), az2);
      float lo, hi;
      unpack2(fma2(dz, dz, fma2(dx, dx, mul2(dy, dy))), lo, hi);
      if (WANT_INDEX) {
        const int i0 = ch * CHUNK + 2 * k;
        if (lo < e || (lo == e && ei != 0x7fffffff && (perm ? perm[i0] < perm[ei] : i0 < ei))) { e = lo; ei = i0; }
        if (hi < e || (hi == e && ei != 0x7fffffff && (perm ? perm[i0 + 1] < perm[ei] : i0 + 1 < ei))) { e = hi; ei = i0 + 1; }
      } else {
        e = min3(e, lo, hi);
      }
    }
  }
  float m = e;
  #pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fminf(m, __shfl_xor_sync(0xffffffffu, m, o));
  best = m;
  if (WANT_INDEX) {
    const bool mine = e == m && ei != 0x7fffffff;
    const unsigned key = mine ? (unsigned)(perm ? perm[ei] : ei) : 0x7fffffffu;
    const unsigned kmin = __reduce_min_sync(0xffffffffu, key);
    const unsigned who = __ballot_sync(0xffffffffu, mine && key == kmin);
    best_pos = who ? __shfl_sync(0xffffffffu, ei, __ffs(who) - 1) : 0x7fffffff;
  }
}

// One matrix entry from its two directed sums: M[i,j] (+ mirror) and the fused MMD/COV/1-NNA reductions.
__device__ __forceinline__ void emit_entry(const Params& p, int ci, int cj, double S0, double S1) {
  const float v = (float)(S0 / (double)p.countX) + (float)(S1 / (double)p.countY);
  if (p.M) {
    p.M[(long long)(p.compact_rows ? (int)blockIdx.y : ci) * p.ldm + cj] = v;
    if (p.symmetric && p.mirror && ci != cj) p.M[(long long)cj * p.ldm + ci] = v;
  }
  // fused _compute_cov_mmd / _compute_nna(k=1) reductions (reference cov_mmd_1nna.py:54-106): v >= 0, so
  // (bits << 32 | index) orders by value, then by index -- torch's lowest-index tie rule on this path
  if (p.keys) {
    const int gi = p.offX + ci, gj = p.offY + cj;
    if (gi != gj) {                                              // the +inf diagonal of _compute_nna
      const unsigned long long vb = (unsigned long long)__float_as_uint(v) << 32;
      atomicMin(p.keys + gj, vb | (unsigned)gi);
      atomicMin(p.keys + gi, vb | (unsigned)gj);
      const int lo = min(gi, gj), hi = max(gi, gj);
      if (lo < p.n_ref && hi >= p.n_ref) {                       // an entry of M_rg: lo is the reference cloud
        atomicMin(p.keys + p.n_total + hi, vb | (unsigned)lo);
        atomicMin(p.keys + 2 * (long long)p.n_total + lo, vb | (unsigned)hi);
      }
    }
  }
}

// NT threads per CTA. The register tile of R = 8 rows per thread is what makes the search FMA-bound
// (one LDS.128 pair feeds 24 FFMA2), so small clouds keep R = 8 and shrink the CTA instead: 2048 rows
// -> 256 threads, 1024 -> 128, 512 -> 64, 256 -> 32 (the matrix front end's table, dispatch_matrix). Every
// shape keeps 16 warps of 128 registers per SM; the R < 8 instantiations (batch front end on small
// batches, odd sizes) trade registers for residency because their CTAs are short.
// MERGED: merged-origin clouds (prep_merge_kernel) too large for the sort, in the matrix front end.
template <int R, bool MATRIX, bool MERGED, int NT = TPB>
__global__ void __launch_bounds__(NT, R >= 8 ? 512 / NT : (R == 4 ? 3 : 4)) nn_kernel(const Params p) {
  static_assert(!MERGED || MATRIX, "merged origins are a matrix front end layout");
  extern __shared__ __align__(128) unsigned char smem_raw[];
  float4* const tiles = reinterpret_cast<float4*>(smem_raw);
  __shared__ uint64_t bars[2];
  __shared__ double red[NT / 32];

  constexpr int RB = NT * R;
  // candidates per search chunk = the window the exact pass re-evaluates per row and tile. Small clouds (the
  // shrunken CTAs) take 16: the exact pass is a fixed cost per row, 14 % of the search at 512 points with 32.
  constexpr int CH = (NT < TPB && !MERGED) ? CHUNK / 2 : CHUNK;      // merged clouds: the DEFERRED pass reads whole chunks
  constexpr int PR = CH / 2;
  const int tid = threadIdx.x;
  const int lane = tid & 31;

  // ---- which clouds ----
  int ci, cj;            // cloud index on the X side and on the Y side
  int dir_only = -1, rb_only = 0;
  if (MATRIX) {
    ci = p.row_begin + blockIdx.y * p.row_stride;
    cj = blockIdx.x;
    if (p.symmetric && cj < ci) return;
  } else {
    ci = cj = blockIdx.y;
    dir_only = blockIdx.z;
    rb_only = blockIdx.x;
    const int rows_here = dir_only == 0 ? p.countX : p.countY;
    if (rb_only >= (rows_here + RB - 1) / RB) return;
  }
  const float4* const sx = p.scanX + (long long)ci * p.strideX;
  const float4* const sy = p.scanY + (long long)cj * p.strideY;

  // points actually scanned per cloud; with merged origins the last one stands for `wlast` identical
  // (0,0,0) points of the original cloud (SURVEY.md S7: means still divide by the full count)
  int2 mx = make_int2(p.countX, 1), my = make_int2(p.countY, 1);
  if (MERGED) { mx = p.metaX[ci]; my = p.metaY[cj]; }
// Merged clouds have arbitrary point counts, so the last row block of a direction is usually almost empty
// (16 390 points = 8 full blocks + 6 rows). There a warp owns 32 R consecutive rows, and a warp without
// live rows skips the search: the FMA pipe it would have occupied goes to the SM's other resident CTA.
#define K_ROW(r) (MERGED ? rb * RB + (tid >> 5) * (32 * R) + (r) * 32 + lane : rb * RB + (r) * NT + tid)
#define K_countX (MERGED ? mx.x : p.countX)
#define K_countY (MERGED ? my.x : p.countY)
#define K_paddedX (MERGED ? (mx.x + CHUNK - 1) / CHUNK * CHUNK : p.paddedX)
#define K_paddedY (MERGED ? (my.x + CHUNK - 1) / CHUNK * CHUNK : p.paddedY)

  const int ntX = (K_paddedX + TILE - 1) / TILE, ntY = (K_paddedY + TILE - 1) / TILE;
  const int nrbX = (K_countX + RB - 1) / RB, nrbY = (K_countY + RB - 1) / RB;
  const int seg0 = nrbX * ntY;
  int pos_begin, pos_end;
  if (MATRIX) { pos_begin = 0; pos_end = seg0 + nrbY * ntX; }
  else if (dir_only == 0) { pos_begin = rb_only * ntY; pos_end = pos_begin + ntY; }
  else { pos_begin = seg0 + rb_only * ntX; pos_end = pos_begin + ntX; }

  // the two tile buffers are as large as the largest tile of this launch (launch_nn sizes the dynamic shared
  // memory the same way): small clouds leave room for more resident CTAs to hide the per-entry prologue
  const int tstride = (R >= 8 && NT == TPB) ? TILE : min(TILE, max(p.paddedX, p.paddedY));
  if (tid == 0) { mbar_init(&bars[0], 1); mbar_init(&bars[1], 1); mbar_fence_init(); }
  __syncthreads();

  // tile stream: position -> (direction, scan tile)
  auto issue = [&](int pos, int buf) {
    int dir, t;
    if (pos < seg0) { dir = 0; t = pos % ntY; } else { dir = 1; t = (pos - seg0) % ntX; }
    const float4* src = (dir == 0 ? sy : sx) + (long long)t * TILE;
    const int padded = dir == 0 ? K_paddedY : K_paddedX;
    const int npts = min(TILE, padded - t * TILE);
    mbar_expect_tx(&bars[buf], (uint32_t)npts * 16u);
    bulk_g2s(tiles + buf * tstride, src, (uint32_t)npts * 16u, &bars[buf]);
  };
  if (tid == 0) issue(pos_begin, 0);

  f32x2 nax[R], nay[R], naz[R];     // {-2a, -2a}: search operands; ptxas folds the pair into FFMA2's scalar-broadcast form
  float eb[R];                      // exact running minimum over tiles
  int ei[R];                        // its index (batch front end only)
  // search state: best and runner-up chunk minima of |b|^2 - 2 a.b and the best chunk's number. Dense clouds
  // restart it for every tile (the exact pass follows the tile); merged clouds carry it across all tiles of a row
  // block and defer the exact pass to the end (see DEFERRED below).
  float cur[R], sec[R];
  int cid[R];
  double dsum = 0.0, S0 = 0.0;

  for (int pos = pos_begin; pos < pos_end; ++pos) {
    const int it = pos - pos_begin;
    const int buf = it & 1;
    if (tid == 0 && pos + 1 < pos_end) issue(pos + 1, buf ^ 1);

    int dir, rb, t, nt;
    if (pos < seg0) { dir = 0; rb = pos / ntY; t = pos - rb * ntY; nt = ntY; }
    else { dir = 1; const int q = pos - seg0; rb = q / ntX; t = q - rb * ntX; nt = ntX; }
    const float4* const rows = dir == 0 ? sx : sy;
    const int rowcount = dir == 0 ? K_countX : K_countY;
    const int scanpadded = dir == 0 ? K_paddedY : K_paddedX;

    if (t == 0) {
      #pragma unroll
      for (int r = 0; r < R; ++r) {
        const int row = K_ROW(r);
        const int rr = row < rowcount ? row : 0;
        const float4 a0 = rows[(rr >> 1) * 2], a1 = rows[(rr >> 1) * 2 + 1];
        const bool hi = rr & 1;
        const float mx = -2.0f * (hi ? a0.y : a0.x), my = -2.0f * (hi ? a0.w : a0.z), mz = -2.0f * (hi ? a1.y : a1.x);
        nax[r] = pack2(mx, mx);
        nay[r] = pack2(my, my);
        naz[r] = pack2(mz, mz);
        eb[r] = __int_as_float(0x7f800000);
        ei[r] = 0;
        if (MERGED) { cur[r] = sec[r] = __int_as_float(0x7f800000); cid[r] = 0; }
      }
    }

    mbar_wait(&bars[buf], (uint32_t)((it >> 1) & 1));
    const float4* const tp = tiles + buf * tstride;
    const int nch = min(TILE, scanpadded - t * TILE) / CH;

    if (!MERGED || rb * RB + (tid >> 5) * (32 * R) < rowcount) {      // warp-uniform
    // ---- search: which chunk of this tile holds the smallest |b|^2 - 2 a.b ----
    if (!MERGED) {
      #pragma unroll
      for (int r = 0; r < R; ++r) { cur[r] = sec[r] = __int_as_float(0x7f800000); cid[r] = 0; }
    }
    const int cbase = MERGED ? t * (TILE / CH) : 0;      // merged clouds number their chunks through the whole cloud
    for (int c = 0; c < nch; ++c) {
      const float4* cp = tp + c * CH;
      float cm[R];
      #pragma unroll
      for (int k = 0; k < PR; ++k) {
        const float4 q0 = cp[2 * k], q1 = cp[2 * k + 1];
        const f32x2 bx = pack2(q0.x, q0.y), by = pack2(q0.z, q0.w);
        const f32x2 bz = pack2(q1.x, q1.y), bn = pack2(q1.z, q1.w);
        #pragma unroll
        for (int r = 0; r < R; ++r) {
          f32x2 s = fma2(naz[r], bz, bn);
          s = fma2(nay[r], by, s);
          s = fma2(nax[r], bx, s);
          float lo, hi;
          unpack2(s, lo, hi);
          cm[r] = (k == 0) ? fminf(lo, hi) : min3(cm[r], lo, hi);
        }
      }
      #pragma unroll
      for (int r = 0; r < R; ++r) {
        const bool better = cm[r] < cur[r];     // strict: the earliest chunk keeps bit-equal minima
        sec[r] = fminf(sec[r], better ? cur[r] : cm[r]);      // runner-up: the smallest minimum of any other chunk
        cur[r] = better ? cm[r] : cur[r];
        cid[r] = better ? cbase + c : cid[r];
      }
    }

    if (MERGED && p.visited != nullptr && lane == 0) {          // bench.py's executed-flop count for pruned workloads
      const int first = rb * RB + (tid >> 5) * (32 * R);
      atomicAdd(p.visited, (unsigned long long)nch * CH * (unsigned long long)min(32 * R, rowcount - first));
    }
    // ---- exact: re-evaluate the winning chunk with the reference's rounding ----
    constexpr int G = R < 4 ? R : 4;
    if (!MERGED)                          // merged clouds: once per row block, after the last tile (DEFERRED)
    #pragma unroll
    for (int g = 0; g < R; g += G) {
      float e[G];
      int eidx[G];
      f32x2 ax2[G], ay2[G], az2[G];
      const float4* cp[G];
      #pragma unroll
      for (int r = 0; r < G; ++r) {
        e[r] = __int_as_float(0x7f800000);
        eidx[r] = 0x7fffffff;
        const f32x2 mh = pack2(-0.5f, -0.5f);      // exact: recovers the row point from -2a
        ax2[r] = mul2(nax[g + r], mh); ay2[r] = mul2(nay[g + r], mh); az2[r] = mul2(naz[g + r], mh);
        cp[r] = tp + cid[g + r] * CH;
      }
      #pragma unroll 4
      for (int k = 0; k < PR; ++k) {
        const int kk = (k + lane) & (PR - 1);   // lanes start on different banks
        #pragma unroll
        for (int r = 0; r < G; ++r) {
          const float4 q0 = cp[r][2 * kk], q1 = cp[r][2 * kk + 1];
          const f32x2 dx = sub2(pack2(q0.x, q0.y), ax2[r]);
          const f32x2 dy = sub2(pack2(q0.z, q0.w), ay2[r]);
          const f32x2 dz = sub2(pack2(q1.x, q1.y), az2[r]);
          const f32x2 d = fma2(dz, dz, fma2(dx, dx, mul2(dy, dy)));
          float lo, hi;
          unpack2(d, lo, hi);
          if (MATRIX) {
            e[r] = min3(e[r], lo, hi);
          } else {
            const int i0 = t * TILE + cid[g + r] * CH + 2 * kk;
            if (lo < e[r] || (lo == e[r] && (eidx[r] == 0x7fffffff || i0 < eidx[r]))) { e[r] = lo; eidx[r] = i0; }
            if (hi < e[r] || (hi == e[r] && (eidx[r] == 0x7fffffff || i0 + 1 < eidx[r]))) { e[r] = hi; eidx[r] = i0 + 1; }
          }
        }
      }
      #pragma unroll
      for (int r = 0; r < G; ++r) {
        if (MATRIX) {
          eb[g + r] = fminf(eb[g + r], e[r]);
        } else if (e[r] < eb[g + r]) {
          eb[g + r] = e[r];                        // tiles ascend, so the lowest index keeps ties by itself
          ei[g + r] = eidx[r];
        }
      }
    }

    // ---- guard: a runner-up chunk inside the search's error window => the whole tile, exactly, for that row ----
    if (!MERGED) {
      #pragma unroll
      for (int r = 0; r < R; ++r) {
        float ax, ay, az, dummy;
        unpack2(nax[r], ax, dummy); unpack2(nay[r], ay, dummy); unpack2(naz[r], az, dummy);
        ax *= -0.5f; ay *= -0.5f; az *= -0.5f;
        const bool near_tie = K_ROW(r) < rowcount && sec[r] <= cur[r] + search_window(ax, ay, az, cur[r]);
        unsigned flagged = __ballot_sync(0xffffffffu, near_tie);
        while (flagged) {                         // warp-uniform; ~0.1 % of the (row, tile) pairs on LiDAR-like clouds
          const int src = __ffs(flagged) - 1;
          flagged &= flagged - 1;
          float m;
          int mi = 0;
          warp_tile_exact_min<!MATRIX>(tp, nch * PR, __shfl_sync(0xffffffffu, ax, src), __shfl_sync(0xffffffffu, ay, src),
                                       __shfl_sync(0xffffffffu, az, src), lane, m, mi);
          if (lane == src) {
            if (MATRIX) {
              eb[r] = fminf(eb[r], m);
            } else if (mi != 0x7fffffff) {
              mi += t * TILE;
              if (m < eb[r] || (m == eb[r] && mi < ei[r])) { eb[r] = m; ei[r] = mi; }
            }
          }
        }
      }
    }

    }

    // ---- DEFERRED (merged clouds): after the last tile of a row block, the exact pass on each row's winning chunk
    //      and the guard over the whole cloud, both straight from global memory (L2): once per row block instead
    //      of once per tile ----
    if (MERGED && t == nt - 1 && rb * RB + (tid >> 5) * (32 * R) < rowcount) {      // warp-uniform
      const float4* const cand = dir == 0 ? sy : sx;
      #pragma unroll
      for (int r = 0; r < R; ++r) {
        float ax, ay, az, dummy;
        unpack2(nax[r], ax, dummy); unpack2(nay[r], ay, dummy); unpack2(naz[r], az, dummy);
        ax *= -0.5f; ay *= -0.5f; az *= -0.5f;
        const bool live = K_ROW(r) < rowcount;
        float e = __int_as_float(0x7f800000);
        if (live && cur[r] < __int_as_float(0x7f800000)) {
          const f32x2 ax2 = pack2(ax, ax), ay2 = pack2(ay, ay), az2 = pack2(az, az);
          const float4* cp = cand + (long long)cid[r] * CHUNK;
          #pragma unroll 4
          for (int k = 0; k < CHUNK / 2; ++k) {
            const float4 q0 = cp[2 * k], q1 = cp[2 * k + 1];
            const f32x2 dx = sub2(pack2(q0.x, q0.y), ax2);
            const f32x2 dy = sub2(pack2(q0.z, q0.w), ay2);
            const f32x2 dz = sub2(pack2(q1.x, q1.y), az2);
            float lo, hi;
            unpack2(fma2(dz, dz, fma2(dx, dx, mul2(dy, dy))), lo, hi);
            e = min3(e, lo, hi);
          }
        }
        eb[r] = e;
        const bool near_tie = live && sec[r] <= cur[r] + search_window(ax, ay, az, cur[r]);
        unsigned flagged = __ballot_sync(0xffffffffu, near_tie);
        while (flagged) {                         // warp-uniform
          const int src = __ffs(flagged) - 1;
          flagged &= flagged - 1;
          float m;
          int mi;
          warp_cloud_exact_min<false>(cand, scanpadded / CHUNK, nullptr, 0.0f, __shfl_sync(0xffffffffu, ax, src),
                                      __shfl_sync(0xffffffffu, ay, src), __shfl_sync(0xffffffffu, az, src), lane, nullptr, m, mi);
          if (lane == src) eb[r] = fminf(eb[r], m);
        }
      }
    }

    // ---- end of a (direction, row block): emit ----
    if (t == nt - 1) {
      #pragma unroll
      for (int r = 0; r < R; ++r) {
        const int row = K_ROW(r);
        if (row < rowcount) {
          if (MATRIX) {
            if (MERGED) dsum += (row == rowcount - 1 ? (double)(dir == 0 ? mx.y : my.y) : 1.0) * (double)eb[r];
            else dsum += (double)eb[r];
          } else {
            float* dist = dir == 0 ? p.dist1 : p.dist2;
            int* idx = dir == 0 ? p.idx1 : p.idx2;
            const long long o = (long long)ci * rowcount + row;
            dist[o] = eb[r];
            if (idx) idx[o] = ei[r] == 0x7fffffff ? 0 : ei[r];
          }
        }
      }
    }
    if (MATRIX && pos == seg0 - 1) { S0 = block_sum<NT>(dsum, red); dsum = 0.0; }
    __syncthreads();   // everyone is done with tiles[buf] before it is refilled
  }

  if (MATRIX) {
    const double S1 = block_sum<NT>(dsum, red);
    if (tid == 0) emit_entry(p, ci, cj, S0, S1);
  }
}

#undef K_ROW
#undef K_countX
#undef K_countY
#undef K_paddedX
#undef K_paddedY

// xyz (clouds, count, 3) -> scan format (clouds, padded/2, 2) float4; padding is NaN so that it
// never wins a min (FMNMX returns the non-NaN operand).
__global__ void __launch_bounds__(256) prep_kernel(const float* __restrict__ xyz, long long clouds, int count,
                                                   int padded, float4* __restrict__ out) {
  const long long half = padded / 2;
  const long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= clouds * half) return;
  const long long c = g / half;
  const int q = (int)(g - c * half);
  const float nan = __int_as_float(0x7fc00000);
  float v[2][4];
  #pragma unroll
  for (int s = 0; s < 2; ++s) {
    const int pt = 2 * q + s;
    if (pt < count) {
      const float* src = xyz + (c * count + pt) * 3;
      const float x = src[0], y = src[1], z = src[2];
      v[s][0] = x; v[s][1] = y; v[s][2] = z;
      v[s][3] = fmaf(z, z, fmaf(x, x, y * y));
    } else {
      v[s][0] = v[s][1] = v[s][2] = v[s][3] = nan;
    }
  }
  out[g * 2] = make_float4(v[0][0], v[1][0], v[0][1], v[1][1]);
  out[g * 2 + 1] = make_float4(v[0][2], v[1][2], v[0][3], v[1][3]);
}

// Scan format with merged origins (one CTA per cloud): the points that are not exactly (0,0,0) keep
// their order, all (0,0,0) points -- dropped pixels of an un-sampled cloud, SURVEY.md S7 -- collapse
// into ONE origin point appended last, whose multiplicity goes to meta[c].y. A nearest-neighbour
// minimum does not depend on duplicate candidates and identical rows have identical minima, so the
// sums over the original cloud are recovered exactly by weighting that row.
__global__ void __launch_bounds__(256) prep_merge_kernel(const float* __restrict__ xyz, int count, long long stride,
                                                         float4* __restrict__ out, int2* __restrict__ meta) {
  __shared__ int wsum[8];
  const long long c = blockIdx.x;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const float* src = xyz + c * count * 3;
  float* dst = reinterpret_cast<float*>(out + c * stride);
  const int per = (count + 255) / 256;                // consecutive points per thread: order is preserved
  const int begin = min(tid * per, count), end = min(begin + per, count);
  int mine = 0;
  for (int i = begin; i < end; ++i) mine += (src[3 * i] != 0.0f) || (src[3 * i + 1] != 0.0f) || (src[3 * i + 2] != 0.0f);
  int inc = mine;
  #pragma unroll
  for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += t; }
  if (lane == 31) wsum[warp] = inc;
  __syncthreads();
  int before = 0, total = 0;
  #pragma unroll
  for (int w = 0; w < 8; ++w) { if (w < warp) before += wsum[w]; total += wsum[w]; }
  auto put = [&](int pos, float x, float y, float z, float n) {
    float* q = dst + (size_t)(pos >> 1) * 8 + (pos & 1);     // {x0,x1,y0,y1}{z0,z1,n0,n1}
    q[0] = x; q[2] = y; q[4] = z; q[6] = n;
  };
  int pos = before + inc - mine;
  for (int i = begin; i < end; ++i) {
    const float x = src[3 * i], y = src[3 * i + 1], z = src[3 * i + 2];
    if (x != 0.0f || y != 0.0f || z != 0.0f) put(pos++, x, y, z, fmaf(z, z, fmaf(x, x, y * y)));
  }
  const int zeros = count - total;
  const int kept = total + (zeros > 0 ? 1 : 0);
  if (tid == 0) {
    if (zeros > 0) put(total, 0.0f, 0.0f, 0.0f, 0.0f);
    meta[c] = make_int2(kept, zeros > 0 ? zeros : 1);
  }
  const float nan = __int_as_float(0x7fc00000);
  const int padded = (kept + CHUNK - 1) / CHUNK * CHUNK;
  for (int i = kept + tid; i < padded; i += 256) put(i, nan, nan, nan, nan);
}

// Merged origins + spatial order (clouds of at most SORT_CAP points): the kept points are sorted by a
// Morton cell key (x, y interleaved at 7 bits each, z 1 bit, ties by original index, so the order is
// deterministic) or into k-d order (below) with bitonic networks in shared memory, written in scan format,
// and every 32-candidate chunk and every block of 32 chunks gets its bounding box. The pair and walk kernels
// skip a chunk whenever the gap between the chunk's box and a row or a row group's box is already no smaller
// than the current minima of those rows: exact, because every operation of the distance is monotone in
// |dx|,|dy|,|dz| and so is rounding.
constexpr int SORT_CAP = 32768;
constexpr int SORT_TPB = 1024;
constexpr int WALK_BLOCKS = SORT_CAP / CHUNK / 32;      // blocks of 32 chunks per cloud (upper level of the best-first walk)

__device__ __forceinline__ unsigned spread7(unsigned v) {          // abcdefg -> a0b0c0d0e0f0g
  v &= 0x7fu;
  v = (v | (v << 4)) & 0x070fu;
  v = (v | (v << 2)) & 0x1333u;
  v = (v | (v << 1)) & 0x1555u;
  return v;
}

// float -> unsigned with the same order (for shared-memory atomicMin / atomicMax on coordinates), and back
__device__ __forceinline__ unsigned ordered_bits(float f) {
  const unsigned u = __float_as_uint(f);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float ordered_float(unsigned u) {
  return __uint_as_float((u & 0x80000000u) ? (u & 0x7fffffffu) : ~u);
}

// KD = false: Morton order (one sort). KD = true: k-d order -- the cloud is split in two halves along the widest axis
// of its bounding box, each half along the widest axis of ITS box, and so on down to the 32-point chunks: chunks are
// the leaves of a balanced k-d tree, their boxes are disjoint and tight whatever the density (Morton cells on a
// uniform grid give chunks that straddle cells: LiDAR clouds are dense near the sensor and sparse far away), and a
// run of 2^k chunks is a subtree with a tight box of its own. One segmented bitonic sort per level; splits sit at
// power-of-two positions, the padding stays a suffix of the last non-empty segment at every level.
constexpr int KD_MAXSEG = SORT_CAP / 64;
// NT threads per CTA: 1024 for large clouds (one CTA per SM: the keys take up to 128 KB), 256 for clouds of at most 4096
// points, where several CTAs per SM hide the latency of the per-level passes (2000 clouds of 2048 points: 1.17 -> 0.72 ms)
// One launch sorts the clouds of up to two sets (the X and Y sides of a call: CTAs [0, clouds0) take side 0, the others side 1),
// so that the two sides of a small batch share the GPU instead of running one after the other.
struct SortSide {
  const float* xyz; int count; long long stride; float4* out; int2* meta; float4* boxes; int boxstride;
  int* perm; int* inv; float4* block_boxes;
};
struct SortArgs { SortSide s[2]; int clouds0; };

template <bool KD, int NT>
__global__ void __launch_bounds__(NT, NT == 1024 ? 1 : 6) prep_sort_kernel(const SortArgs a) {
  extern __shared__ unsigned keys[];            // n2 keys (next power of two >= count)
  __shared__ float red[NT / 32][6];
  __shared__ int wsum[NT / 32];
  __shared__ int first_zero;
  const bool side = (int)blockIdx.x >= a.clouds0;
  const long long c = (int)blockIdx.x - (side ? a.clouds0 : 0);
  const float* __restrict__ const xyz = side ? a.s[1].xyz : a.s[0].xyz;
  const int count = side ? a.s[1].count : a.s[0].count;
  const long long stride = side ? a.s[1].stride : a.s[0].stride;
  float4* __restrict__ const out = side ? a.s[1].out : a.s[0].out;
  int2* __restrict__ const meta = side ? a.s[1].meta : a.s[0].meta;
  float4* __restrict__ const boxes = side ? a.s[1].boxes : a.s[0].boxes;
  const int boxstride = side ? a.s[1].boxstride : a.s[0].boxstride;
  int* __restrict__ const perm_all = side ? a.s[1].perm : a.s[0].perm;
  int* __restrict__ const inv_all = side ? a.s[1].inv : a.s[0].inv;
  float4* __restrict__ const block_boxes = side ? a.s[1].block_boxes : a.s[0].block_boxes;
  // batch front end only: perm[position] = original index (the merged origin point stands for the FIRST zero point,
  // the arg-min the reference reports among equal distances), inv[original index] = position
  int* const perm = perm_all ? perm_all + c * stride : nullptr;
  int* const inv = inv_all ? inv_all + c * count : nullptr;
  if (threadIdx.x == 0) first_zero = 0x7fffffff;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const float* src = xyz + c * count * 3;
  float* dst = reinterpret_cast<float*>(out + c * stride);
  float4* bdst = boxes + c * boxstride;
  const float inf = __int_as_float(0x7f800000);
  int n2 = 1;
  while (n2 < count) n2 <<= 1;

  // ---- bounding box of the non-zero points, their number ----
  float lo[3] = {inf, inf, inf}, hi[3] = {-inf, -inf, -inf};
  int mine = 0;
  for (int i = tid; i < count; i += NT) {
    const float x = src[3 * i], y = src[3 * i + 1], z = src[3 * i + 2];
    if (x != 0.0f || y != 0.0f || z != 0.0f) {
      ++mine;
      lo[0] = fminf(lo[0], x); lo[1] = fminf(lo[1], y); lo[2] = fminf(lo[2], z);
      hi[0] = fmaxf(hi[0], x); hi[1] = fmaxf(hi[1], y); hi[2] = fmaxf(hi[2], z);
    }
  }
  __syncthreads();                              // first_zero is initialised
  #pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    mine += __shfl_xor_sync(0xffffffffu, mine, o);
    #pragma unroll
    for (int a = 0; a < 3; ++a) {
      lo[a] = fminf(lo[a], __shfl_xor_sync(0xffffffffu, lo[a], o));
      hi[a] = fmaxf(hi[a], __shfl_xor_sync(0xffffffffu, hi[a], o));
    }
  }
  if (lane == 0) {
    wsum[warp] = mine;
    #pragma unroll
    for (int a = 0; a < 3; ++a) { red[warp][a] = lo[a]; red[warp][3 + a] = hi[a]; }
  }
  __syncthreads();
  int total = 0;
  for (int w = 0; w < NT / 32; ++w) {
    total += wsum[w];
    #pragma unroll
    for (int a = 0; a < 3; ++a) { lo[a] = fminf(lo[a], red[w][a]); hi[a] = fmaxf(hi[a], red[w][3 + a]); }
  }
  // k-d order: a lone (0,0,0) point is an ordinary point (FPS samples keep at most one); only two or more collapse
  const bool single = KD && count - total == 1;
  if (single) total = count;
  const float sxs = hi[0] > lo[0] ? 128.0f / (hi[0] - lo[0]) : 0.0f;
  const float sys = hi[1] > lo[1] ? 128.0f / (hi[1] - lo[1]) : 0.0f;
  const float szs = hi[2] > lo[2] ? 2.0f / (hi[2] - lo[2]) : 0.0f;

  if (!KD) {
  // ---- keys: (cell << 15) | original index; zero points and padding sort to the end ----
  for (int i = tid; i < n2; i += NT) {
    unsigned key = 0xffffffffu;
    if (i < count) {
      const float x = src[3 * i], y = src[3 * i + 1], z = src[3 * i + 2];
      if (x != 0.0f || y != 0.0f || z != 0.0f) {
        const unsigned ix = (unsigned)min(127, max(0, (int)((x - lo[0]) * sxs)));
        const unsigned iy = (unsigned)min(127, max(0, (int)((y - lo[1]) * sys)));
        const unsigned iz = (unsigned)min(1, max(0, (int)((z - lo[2]) * szs)));
        key = ((((spread7(ix) | (spread7(iy) << 1)) << 1) | iz) << 15) | (unsigned)i;
      }
    }
    keys[i] = key;
  }
  __syncthreads();
  for (int k = 2; k <= n2; k <<= 1) {
    for (int j = k >> 1; j > 0; j >>= 1) {
      for (int t = tid; t < (n2 >> 1); t += NT) {
        const int i = ((t & ~(j - 1)) << 1) | (t & (j - 1));
        const int l = i | j;
        const unsigned a = keys[i], b = keys[l];
        const bool up = (i & k) == 0;
        if ((a > b) == up) { keys[i] = b; keys[l] = a; }
      }
      __syncthreads();
    }
  }
  } else {
  // ---- k-d order: per level, (position along the segment's widest axis, 17 bits) << 15 | original index ----
  __shared__ unsigned seglo[KD ? 3 * KD_MAXSEG : 1], seghi[KD ? 3 * KD_MAXSEG : 1];
  for (int i = tid; i < n2; i += NT) {
    unsigned key = 0xffffffffu;
    if (i < count && (single || src[3 * i] != 0.0f || src[3 * i + 1] != 0.0f || src[3 * i + 2] != 0.0f)) key = (unsigned)i;
    keys[i] = key;
  }
  // level 0 packs the kept points to the front (its keys carry the global box: one segment)
  for (int seglen = n2; seglen >= 2 * CHUNK || seglen == n2; seglen >>= 1) {      // tiny clouds: one level packs them
    const int nseg = n2 / seglen;
    for (int sgi = tid; sgi < 3 * nseg; sgi += NT) { seglo[sgi] = 0xffffffffu; seghi[sgi] = 0u; }
    __syncthreads();
    for (int base = warp * 32; base < n2; base += NT) {          // 32 consecutive positions: one segment
      const unsigned key = base + lane < n2 ? keys[base + lane] : 0xffffffffu;
      float v[3] = {inf, inf, inf}, w[3] = {-inf, -inf, -inf};
      if (key != 0xffffffffu) {
        const int i = (int)(key & 0x7fffu);
        v[0] = w[0] = src[3 * i]; v[1] = w[1] = src[3 * i + 1]; v[2] = w[2] = src[3 * i + 2];
      }
      if (__any_sync(0xffffffffu, key != 0xffffffffu)) {
        #pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
          #pragma unroll
          for (int a = 0; a < 3; ++a) {
            v[a] = fminf(v[a], __shfl_xor_sync(0xffffffffu, v[a], o));
            w[a] = fmaxf(w[a], __shfl_xor_sync(0xffffffffu, w[a], o));
          }
        }
        const int sg = base / seglen;
        if (lane < 3) atomicMin(&seglo[3 * sg + lane], ordered_bits(lane == 0 ? v[0] : lane == 1 ? v[1] : v[2]));
        else if (lane < 6) atomicMax(&seghi[3 * sg + lane - 3], ordered_bits(lane == 3 ? w[0] : lane == 4 ? w[1] : w[2]));
      }
    }
    __syncthreads();
    for (int pos = tid; pos < n2; pos += NT) {
      const unsigned key = keys[pos];
      if (key == 0xffffffffu) continue;
      const int i = (int)(key & 0x7fffu);
      const int sg = pos / seglen;
      const float l0 = ordered_float(seglo[3 * sg]), l1 = ordered_float(seglo[3 * sg + 1]), l2 = ordered_float(seglo[3 * sg + 2]);
      const float e0 = ordered_float(seghi[3 * sg]) - l0, e1 = ordered_float(seghi[3 * sg + 1]) - l1, e2 = ordered_float(seghi[3 * sg + 2]) - l2;
      const int ax = (e0 >= e1 && e0 >= e2) ? 0 : (e1 >= e2 ? 1 : 2);
      const float ext = ax == 0 ? e0 : ax == 1 ? e1 : e2, base = ax == 0 ? l0 : ax == 1 ? l1 : l2;
      const float q = ext > 0.0f ? (src[3 * i + ax] - base) * (131071.0f / ext) : 0.0f;
      keys[pos] = ((unsigned)min(131070, max(0, (int)q)) << 15) | (unsigned)i;
    }
    __syncthreads();
    for (int k = 2; k <= seglen; k <<= 1) {
      for (int j = k >> 1; j > 0; j >>= 1) {
        for (int t = tid; t < (n2 >> 1); t += NT) {
          const int i = ((t & ~(j - 1)) << 1) | (t & (j - 1));
          const int l = i | j;
          const unsigned a = keys[i], b = keys[l];
          const bool up = (i & k) == 0 || k == seglen;            // every segment ascending
          if ((a > b) == up) { keys[i] = b; keys[l] = a; }
        }
        __syncthreads();
      }
    }
  }
  }

  if (inv != nullptr && !single) {              // zero points: all stand behind the one origin point
    for (int i = tid; i < count; i += NT) {
      if (src[3 * i] == 0.0f && src[3 * i + 1] == 0.0f && src[3 * i + 2] == 0.0f) { inv[i] = total; atomicMin(&first_zero, i); }
    }
    __syncthreads();
  }
  // ---- sorted points in scan format + one origin point + NaN padding; a box per 32-candidate chunk ----
  const int zeros = count - total;
  const int kept = total + (zeros > 0 ? 1 : 0);
  const int padded = (kept + CHUNK - 1) / CHUNK * CHUNK;
  const float nan = __int_as_float(0x7fc00000);
  for (int chunk = warp; chunk < padded / CHUNK; chunk += NT / 32) {
    const int pos = chunk * CHUNK + lane;
    float x = nan, y = nan, z = nan, n = nan;
    if (pos < total) {
      const int i = (int)(keys[pos] & 0x7fffu);
      x = src[3 * i]; y = src[3 * i + 1]; z = src[3 * i + 2];
      n = fmaf(z, z, fmaf(x, x, y * y));
      if (perm) { perm[pos] = i; inv[i] = pos; }
    } else if (pos == total && zeros > 0) {
      x = y = z = n = 0.0f;
      if (perm) perm[pos] = first_zero;
    } else if (perm) {
      perm[pos] = 0;
    }
    float* q = dst + (size_t)(pos >> 1) * 8 + (pos & 1);     // {x0,x1,y0,y1}{z0,z1,n0,n1}
    q[0] = x; q[2] = y; q[4] = z; q[6] = n;
    // the merged origin point stays outside its chunk's box (it would stretch the last leaf's box to the sensor) and
    // the chunk is flagged in .w: the walks always visit it
    const bool sep = zeros > 0;
    const bool real = pos < total;
    float l0 = real ? x : inf, l1 = real ? y : inf, l2 = real ? z : inf;
    float h0 = real ? x : -inf, h1 = real ? y : -inf, h2 = real ? z : -inf;
    #pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      l0 = fminf(l0, __shfl_xor_sync(0xffffffffu, l0, o)); h0 = fmaxf(h0, __shfl_xor_sync(0xffffffffu, h0, o));
      l1 = fminf(l1, __shfl_xor_sync(0xffffffffu, l1, o)); h1 = fmaxf(h1, __shfl_xor_sync(0xffffffffu, h1, o));
      l2 = fminf(l2, __shfl_xor_sync(0xffffffffu, l2, o)); h2 = fmaxf(h2, __shfl_xor_sync(0xffffffffu, h2, o));
    }
    if (lane == 0) {
      bdst[2 * chunk] = make_float4(l0, l1, l2, sep && chunk == padded / CHUNK - 1 ? 1.0f : 0.0f);
      bdst[2 * chunk + 1] = make_float4(h0, h1, h2, 0.f);
    }
  }
  if (tid == 0) meta[c] = make_int2(kept, zeros > 0 ? zeros : 1);
  // ---- boxes of the blocks of 32 chunks (the upper level of nn_walk_split_kernel's best-first walk); empty: (+inf, -inf) ----
  __syncthreads();                              // this CTA's chunk boxes are visible
  float4* const bb = block_boxes + c * (2 * WALK_BLOCKS);
  const int nchunks = padded / CHUNK;
  for (int b = warp; b < WALK_BLOCKS; b += NT / 32) {
    const int chunk = b * 32 + lane;
    float4 bl = make_float4(inf, inf, inf, 0.f), bh = make_float4(-inf, -inf, -inf, 0.f);
    if (chunk < nchunks) { bl = bdst[2 * chunk]; bh = bdst[2 * chunk + 1]; }
    #pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      bl.x = fminf(bl.x, __shfl_xor_sync(0xffffffffu, bl.x, o)); bh.x = fmaxf(bh.x, __shfl_xor_sync(0xffffffffu, bh.x, o));
      bl.y = fminf(bl.y, __shfl_xor_sync(0xffffffffu, bl.y, o)); bh.y = fmaxf(bh.y, __shfl_xor_sync(0xffffffffu, bh.y, o));
      bl.z = fminf(bl.z, __shfl_xor_sync(0xffffffffu, bl.z, o)); bh.z = fmaxf(bh.z, __shfl_xor_sync(0xffffffffu, bh.z, o));
    }
    if (lane == 0) { bb[2 * b] = bl; bb[2 * b + 1] = bh; }
  }
}

// Reference ChamferDistanceGradKernel (chamfer_distance.cu:148-190): after two memsets, every point adds
// 2 g (p - q) to its own gradient and subtracts it from its nearest neighbour's, all with atomicAdd, one launch
// per direction. Here every gradient element is WRITTEN once by the thread that owns the point (its own term, a
// plain 128-bit-friendly store: no memset, no atomic), then one more launch adds the neighbour terms of both
// directions; lanes of a warp that hit the same neighbour are summed in registers first (ordered clouds send
// runs of consecutive points to the same neighbour), so one RED per distinct target leaves the warp.
struct GradArgs {
  int b, n, m;
  const float* xyz1; const float* xyz2;
  const float* gd1; const float* gd2;
  const int* idx1; const int* idx2;
  float* g1; float* g2;
};

// element e of the concatenation [cloud set 1 | cloud set 2] -> (own point, neighbour, 2 g, target slot)
__device__ __forceinline__ bool grad_term(const GradArgs& a, long long e, float (&t)[3], long long& own, long long& nbr, bool& second) {
  const long long n1 = (long long)a.b * a.n, n2 = (long long)a.b * a.m;
  if (e >= n1 + n2) return false;
  second = e >= n1;
  const long long k = second ? e - n1 : e;
  const int cnt = second ? a.m : a.n, other = second ? a.n : a.m;
  const long long i = k / cnt;
  const int j = (second ? a.idx2 : a.idx1)[k];
  const float* p = (second ? a.xyz2 : a.xyz1) + k * 3;
  nbr = i * other + j;
  const float* q = (second ? a.xyz1 : a.xyz2) + nbr * 3;
  const float g = (second ? a.gd2 : a.gd1)[k] * 2.0f;
  t[0] = g * (p[0] - q[0]); t[1] = g * (p[1] - q[1]); t[2] = g * (p[2] - q[2]);
  own = k;
  return true;
}

__global__ void __launch_bounds__(256) grad_own_kernel(const GradArgs a) {
  const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  float t[3]; long long own, nbr; bool second;
  if (!grad_term(a, e, t, own, nbr, second)) return;
  float* o = (second ? a.g2 : a.g1) + own * 3;
  o[0] = t[0]; o[1] = t[1]; o[2] = t[2];
}

__global__ void __launch_bounds__(256) grad_scatter_kernel(const GradArgs a) {
  const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int lane = threadIdx.x & 31;
  float t[3] = {0.f, 0.f, 0.f}; long long own, nbr = -1; bool second = false;
  const bool live = grad_term(a, e, t, own, nbr, second);
  // the neighbour's slot lives in the OTHER gradient; key = slot with the direction in the top bit
  const unsigned long long key = live ? ((unsigned long long)nbr | (second ? 1ull << 62 : 0ull)) : ~0ull - lane;
  const unsigned peers = __match_any_sync(0xffffffffu, key);
  const int leader = __ffs(peers) - 1;
  float sx = t[0], sy = t[1], sz = t[2];
  for (unsigned rest = peers & (peers - 1); rest; rest &= rest - 1) {      // same trip count for every lane of the group
    const int src = __ffs(rest) - 1;
    const float vx = __shfl_sync(peers, t[0], src), vy = __shfl_sync(peers, t[1], src), vz = __shfl_sync(peers, t[2], src);
    if (lane == leader) { sx += vx; sy += vy; sz += vz; }
  }
  if (live && lane == leader) {
    float* o = (second ? a.g1 : a.g2) + nbr * 3;
    atomicAdd(o + 0, -sx); atomicAdd(o + 1, -sy); atomicAdd(o + 2, -sz);
  }
}

static int padded_of(int count) { return (count + CHUNK - 1) / CHUNK * CHUNK; }
static size_t scan_bytes(long long clouds, int count) { return (size_t)clouds * padded_of(count) * 16; }

static int pick_r(int maxcount) {
  if (maxcount > TPB * 4) return 8;
  if (maxcount > TPB * 2) return 4;
  if (maxcount > TPB) return 2;
  return 1;
}

template <int R, bool MATRIX, bool MERGED, int NT = TPB>
static int launch_nn(const Params& p, dim3 grid, cudaStream_t st) {
  static bool configured[kMaxDevices] = {};   // per instantiation and device: the attribute is per context
  const int dev = current_device();
  if (!configured[dev]) {
    DUSTY_CUDA(cudaFuncSetAttribute(nn_kernel<R, MATRIX, MERGED, NT>, cudaFuncAttributeMaxDynamicSharedMemorySize, 2 * TILE * 16));
    configured[dev] = true;
  }
  const int tile_pts = (R >= 8 && NT == TPB) ? TILE : std::min(TILE, std::max(p.paddedX, p.paddedY));
  nn_kernel<R, MATRIX, MERGED, NT><<<grid, NT, 2 * (size_t)tile_pts * 16, st>>>(p);
  DUSTY_AFTER_LAUNCH("chamfer nn_kernel");
  return 0;
}

// Dense matrix front end: (threads per CTA, rows per thread) by cloud size, see nn_kernel.
static int dispatch_matrix(int maxcount, const Params& p, dim3 grid, cudaStream_t st) {
  if (maxcount > 1024) return launch_nn<8, true, false, 256>(p, grid, st);
  if (maxcount > 512) return launch_nn<8, true, false, 128>(p, grid, st);
  if (maxcount > 256) return launch_nn<8, true, false, 64>(p, grid, st);
  if (maxcount > 128) return launch_nn<8, true, false, 32>(p, grid, st);
  return launch_nn<4, true, false, 32>(p, grid, st);
}

// Dense batch front end: R rows per thread, see dusty_chamfer_forward.
static int dispatch_batch(int r, const Params& p, dim3 grid, cudaStream_t st) {
  switch (r) {
    case 8: return launch_nn<8, false, false>(p, grid, st);
    case 4: return launch_nn<4, false, false>(p, grid, st);
    case 2: return launch_nn<2, false, false>(p, grid, st);
    default: return launch_nn<1, false, false>(p, grid, st);
  }
}

static int run_prep(const float* xyz, long long clouds, int count, float4* out, cudaStream_t st) {
  const int padded = padded_of(count);
  const long long work = clouds * (padded / 2);
  if (work == 0) return 0;
  prep_kernel<<<(unsigned)((work + 255) / 256), 256, 0, st>>>(xyz, clouds, count, padded, out);
  DUSTY_AFTER_LAUNCH("chamfer prep_kernel");
  return 0;
}

static size_t meta_bytes(long long clouds) { return align_up((size_t)clouds * sizeof(int2), 256); }

static int run_prep_merge(const float* xyz, long long clouds, int count, float4* out, int2* meta, cudaStream_t st) {
  if (clouds == 0) return 0;
  prep_merge_kernel<<<(unsigned)clouds, 256, 0, st>>>(xyz, count, padded_of(count), out, meta);
  DUSTY_AFTER_LAUNCH("chamfer prep_merge_kernel");
  return 0;
}

static size_t chunk_box_bytes(long long clouds, int count) { return align_up((size_t)clouds * (padded_of(count) / CHUNK) * 32, 256); }
// chunk boxes, then the boxes of the blocks of 32 chunks
static size_t box_bytes(long long clouds, int count) { return chunk_box_bytes(clouds, count) + align_up((size_t)clouds * 2 * WALK_BLOCKS * 16, 256); }
static float4* block_boxes_of(float4* boxes, long long clouds, int count) {
  return reinterpret_cast<float4*>(reinterpret_cast<char*>(boxes) + chunk_box_bytes(clouds, count));
}

// (clouds, count) results at sorted positions -> the original point order (batch front end on sorted clouds)
__global__ void __launch_bounds__(256) unsort_kernel(const float* __restrict__ dist_sorted, const int* __restrict__ idx_sorted,
                                                     const int* __restrict__ inv, long long clouds, int count, long long stride,
                                                     float* __restrict__ dist, int* __restrict__ idx) {
  const long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= clouds * count) return;
  const long long c = g / count;
  const long long o = c * stride + inv[g];
  dist[g] = dist_sorted[o];
  if (idx) idx[g] = idx_sorted[o];
}

static SortSide sort_side(const float* xyz, long long clouds, int count, float4* out, int2* meta, float4* boxes, int* perm, int* inv) {
  return SortSide{xyz, count, (long long)padded_of(count), out, meta, boxes, padded_of(count) / CHUNK * 2, perm, inv,
                  block_boxes_of(boxes, clouds, count)};
}

template <bool KD, int NT>
static int launch_prep_sort(const SortArgs& a, long long clouds, int maxcount, cudaStream_t st) {
  int n2 = 1;
  while (n2 < maxcount) n2 <<= 1;
  static bool configured[kMaxDevices] = {};
  const int dev = current_device();
  if (!configured[dev]) {
    DUSTY_CUDA(cudaFuncSetAttribute(prep_sort_kernel<KD, NT>, cudaFuncAttributeMaxDynamicSharedMemorySize, SORT_CAP * 4));
    configured[dev] = true;
  }
  prep_sort_kernel<KD, NT><<<(unsigned)clouds, NT, (size_t)n2 * 4, st>>>(a);
  DUSTY_AFTER_LAUNCH(KD ? "chamfer prep_sort_kernel<kd>" : "chamfer prep_sort_kernel");
  return 0;
}

// kd: k-d order (Morton otherwise). clouds1 > 0: a second set in the same launch.
static int run_prep_sort2(const SortSide& s0, long long clouds0, const SortSide& s1, long long clouds1, cudaStream_t st, bool kd) {
  if (clouds0 + clouds1 == 0) return 0;
  if (clouds0 + clouds1 > 0x7fffffffLL) return fail_arg(DUSTY_EINVAL, "chamfer: too many clouds in one sort launch");
  SortArgs a{};
  a.s[0] = s0; a.s[1] = clouds1 > 0 ? s1 : s0; a.clouds0 = (int)clouds0;
  const int maxcount = clouds1 > 0 && s1.count > s0.count ? s1.count : s0.count;
  const long long clouds = clouds0 + clouds1;
  if (maxcount <= 4096)
    return kd ? launch_prep_sort<true, 256>(a, clouds, maxcount, st) : launch_prep_sort<false, 256>(a, clouds, maxcount, st);
  return kd ? launch_prep_sort<true, SORT_TPB>(a, clouds, maxcount, st) : launch_prep_sort<false, SORT_TPB>(a, clouds, maxcount, st);
}

#include "chamfer_pair.cuh"
#include "chamfer_walk.cuh"

}  // namespace chamfer
}  // namespace dusty

using namespace dusty;
using namespace dusty::chamfer;

// Measurement only (bench.py, roofline of the pruned workloads): when switched on, the merged-origin kernels add the
// number of (row, candidate) pairs they really evaluate to a device counter.
static unsigned long long* g_visited_counter = nullptr;


// Un-sampled clouds in the batch front end (compute_cd on (B, H*W, 3) pairs, reference evaluate_reconstruction.py:
// 124-131): the same treatment as the matrix front end -- zero points merged into one candidate, kept points
// Morton-sorted with a box per chunk, chunks pruned by box distance -- plus the maps back to the original order.
constexpr int BATCH_SORT_ABOVE = 4096;
static bool forward_takes_sorted_path(int n, int m) {
  const int big = n > m ? n : m;
  return big > BATCH_SORT_ABOVE && big <= SORT_CAP;
}

namespace {
struct SortedSide {          // workspace of one side of a sorted batch call
  float4* scan; int2* meta; float4* boxes; int* perm; int* inv; float* dist; int* idx;
  static size_t bytes(long long b, int count) {
    const size_t pad = (size_t)b * padded_of(count);
    return align_up(scan_bytes(b, count), 256) + meta_bytes(b) + box_bytes(b, count) + 3 * align_up(pad * 4, 256) +
           align_up((size_t)b * count * 4, 256);
  }
  char* carve(char* w, long long b, int count) {
    const size_t pad = (size_t)b * padded_of(count);
    scan = reinterpret_cast<float4*>(w); w += align_up(scan_bytes(b, count), 256);
    meta = reinterpret_cast<int2*>(w); w += meta_bytes(b);
    boxes = reinterpret_cast<float4*>(w); w += box_bytes(b, count);
    perm = reinterpret_cast<int*>(w); w += align_up(pad * 4, 256);
    dist = reinterpret_cast<float*>(w); w += align_up(pad * 4, 256);
    idx = reinterpret_cast<int*>(w); w += align_up(pad * 4, 256);
    inv = reinterpret_cast<int*>(w); w += align_up((size_t)b * count * 4, 256);
    return w;
  }
};
}  // namespace

extern "C" size_t dusty_chamfer_forward_workspace_bytes(int b, int n, int m) {
  if (b <= 0 || n <= 0 || m <= 0) return 0;
  if (forward_takes_sorted_path(n, m)) return SortedSide::bytes(b, n) + SortedSide::bytes(b, m);
  return align_up(scan_bytes(b, n), 256) + align_up(scan_bytes(b, m), 256);
}

extern "C" int dusty_chamfer_forward(const float* xyz1, const float* xyz2, int b, int n, int m, float* dist1,
                                     float* dist2, int32_t* idx1, int32_t* idx2, void* workspace,
                                     size_t workspace_bytes, void* stream) {
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (b < 0 || n < 0 || m < 0) return fail_arg(DUSTY_EINVAL, "chamfer_forward: negative size b=%d n=%d m=%d", b, n, m);
  if (b == 0) return 0;
  if (int rc = check_device()) return rc;
  if (n == 0 || m == 0) {   // the reference leaves its pre-zeroed outputs untouched
    if (n) { DUSTY_CUDA(cudaMemsetAsync(dist1, 0, sizeof(float) * b * n, st)); if (idx1) DUSTY_CUDA(cudaMemsetAsync(idx1, 0, sizeof(int) * b * n, st)); }
    if (m) { DUSTY_CUDA(cudaMemsetAsync(dist2, 0, sizeof(float) * b * m, st)); if (idx2) DUSTY_CUDA(cudaMemsetAsync(idx2, 0, sizeof(int) * b * m, st)); }
    return 0;
  }
  if (!xyz1 || !xyz2 || !dist1 || !dist2 || !workspace) return fail_arg(DUSTY_EINVAL, "chamfer_forward: null pointer");
  if (b > 65535) return fail_arg(DUSTY_EINVAL, "chamfer_forward: batch %d exceeds 65535", b);
  if (!aligned16(workspace)) return fail_arg(DUSTY_EALIGN, "chamfer_forward: workspace must be 16-byte aligned");
  if (workspace_bytes < dusty_chamfer_forward_workspace_bytes(b, n, m))
    return fail_arg(DUSTY_ENOSPACE, "chamfer_forward: workspace %zu < %zu", workspace_bytes,
                    dusty_chamfer_forward_workspace_bytes(b, n, m));
  if (forward_takes_sorted_path(n, m)) {
    SortedSide X, Y;
    Y.carve(X.carve(static_cast<char*>(workspace), b, n), b, m);
    // Order of the batch front end's clouds: each is searched once, so the sort is most of the call. Measured, 8 / 32 / 128 pairs
    // of 32768-point scans with 64-row walk groups: Morton 0.96 / 1.19 / 2.27 ms, k-d 3.45 / 3.52 / 4.12 ms (the k-d sort alone
    // is 1.56 ms per launch: ten segmented sorts); Morton with the 32-row groups of the split walk: 0.78 / 1.04 / 2.02 ms. The
    // matrix front end, where a cloud is searched 2 N times, takes the k-d order.
    if (int rc = run_prep_sort2(sort_side(xyz1, b, n, X.scan, X.meta, X.boxes, X.perm, X.inv), b,
                                sort_side(xyz2, b, m, Y.scan, Y.meta, Y.boxes, Y.perm, Y.inv), b, st, false)) return rc;
    Params p{};
    p.scanX = X.scan; p.scanY = Y.scan;
    p.countX = n; p.countY = m;
    p.paddedX = padded_of(n); p.paddedY = padded_of(m);
    p.strideX = p.paddedX; p.strideY = p.paddedY;
    p.dist1 = X.dist; p.dist2 = Y.dist; p.idx1 = X.idx; p.idx2 = Y.idx;
    p.metaX = X.meta; p.metaY = Y.meta; p.boxX = X.boxes; p.boxY = Y.boxes; p.permX = X.perm; p.permY = Y.perm;
    p.bbX = block_boxes_of(X.boxes, b, n); p.bbY = block_boxes_of(Y.boxes, b, m);
    p.visited = g_visited_counter;
    const int tasks = (n + 31) / 32 + (m + 31) / 32 + 2;      // 32-row groups of both directions (+ the merged origin rows)
    if (int rc = launch_walk_split<false>(p, dim3((tasks + WALK_TPC - 1) / WALK_TPC, b, 1), st)) return rc;
    unsort_kernel<<<(unsigned)(((long long)b * n + 255) / 256), 256, 0, st>>>(X.dist, X.idx, X.inv, b, n, p.strideX, dist1, idx1);
    DUSTY_AFTER_LAUNCH("chamfer unsort_kernel");
    unsort_kernel<<<(unsigned)(((long long)b * m + 255) / 256), 256, 0, st>>>(Y.dist, Y.idx, Y.inv, b, m, p.strideY, dist2, idx2);
    DUSTY_AFTER_LAUNCH("chamfer unsort_kernel");
    return 0;
  }
  float4* s1 = static_cast<float4*>(workspace);
  float4* s2 = reinterpret_cast<float4*>(static_cast<char*>(workspace) + align_up(scan_bytes(b, n), 256));
  if (int rc = run_prep(xyz1, b, n, s1, st)) return rc;
  if (int rc = run_prep(xyz2, b, m, s2, st)) return rc;
  Params p{};
  p.scanX = s1; p.scanY = s2;
  p.countX = n; p.countY = m;
  p.paddedX = padded_of(n); p.paddedY = padded_of(m);
  p.strideX = p.paddedX; p.strideY = p.paddedY;
  p.dist1 = dist1; p.dist2 = dist2; p.idx1 = idx1; p.idx2 = idx2;
  // rows per thread: the largest R that still gives about one CTA per SM (a CTA covers 256 R rows of one
  // direction of one pair); few pairs of small clouds otherwise leave most of the GPU idle. Measured
  // (32 pairs of 2048 points): R = 8 (64 CTAs) 133 us, R = 4 (128 CTAs) 91 us,
  // R = 1 (512 CTAs) 117 us -- smaller R feeds fewer FFMA2 per LDS, so stop as soon as the GPU is covered.
  const int big = n > m ? n : m;
  int r = pick_r(big);
  while (r > 1 && 2LL * b * ((big + TPB * r - 1) / (TPB * r)) < 120) r >>= 1;
  const int rbmax = (big + TPB * r - 1) / (TPB * r);
  return dispatch_batch(r, p, dim3(rbmax, b, 2), st);
}

extern "C" size_t dusty_chamfer_backward_workspace_bytes(int, int, int) { return 0; }

extern "C" int dusty_chamfer_backward(const float* xyz1, const float* xyz2, int b, int n, int m,
                                      const float* grad_dist1, const float* grad_dist2, const int32_t* idx1,
                                      const int32_t* idx2, float* grad_xyz1, float* grad_xyz2, void*, size_t,
                                      void* stream) {
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (b < 0 || n < 0 || m < 0) return fail_arg(DUSTY_EINVAL, "chamfer_backward: negative size");
  if (b == 0) return 0;
  if (int rc = check_device()) return rc;
  if (n == 0 || m == 0) {            // no neighbours: the reference's memsets are all that happens
    if (n) DUSTY_CUDA(cudaMemsetAsync(grad_xyz1, 0, sizeof(float) * 3 * b * n, st));
    if (m) DUSTY_CUDA(cudaMemsetAsync(grad_xyz2, 0, sizeof(float) * 3 * b * m, st));
    return 0;
  }
  if (!xyz1 || !xyz2 || !grad_dist1 || !grad_dist2 || !idx1 || !idx2 || !grad_xyz1 || !grad_xyz2)
    return fail_arg(DUSTY_EINVAL, "chamfer_backward: null pointer");
  const GradArgs a{b, n, m, xyz1, xyz2, grad_dist1, grad_dist2, idx1, idx2, grad_xyz1, grad_xyz2};
  const long long total = (long long)b * n + (long long)b * m;
  const unsigned grid = (unsigned)((total + 255) / 256);
  grad_own_kernel<<<grid, 256, 0, st>>>(a);
  DUSTY_AFTER_LAUNCH("chamfer grad_own_kernel");
  grad_scatter_kernel<<<grid, 256, 0, st>>>(a);
  DUSTY_AFTER_LAUNCH("chamfer grad_scatter_kernel");
  return 0;
}

extern "C" size_t dusty_chamfer_matrix_workspace_bytes(int na, int pa, int nb, int pb) {
  size_t s = 0;
  if (na > 0 && pa > 0) s += align_up(scan_bytes(na, pa), 256) + meta_bytes(na) + box_bytes(na, pa);
  if (nb > 0 && pb > 0) s += align_up(scan_bytes(nb, pb), 256) + meta_bytes(nb) + box_bytes(nb, pb);
  return s;
}

namespace {
struct FusedKeys {            // fused MMD/COV/1-NNA epilogue of the matrix launch (null keys: off)
  unsigned long long* keys = nullptr;
  int n_total = 0, n_ref = 0, off_a = 0, off_b = 0;
};
}  // namespace

static int matrix_impl(const float* A, int na, int pa, const float* B, int nb, int pb, int row_begin, int row_end,
                       int row_stride, int flags, float* M, long long ldm, const FusedKeys& fk, void* workspace,
                       size_t workspace_bytes, void* stream) {
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int symmetric = (flags & DUSTY_MATRIX_SYMMETRIC) != 0, mirror = (flags & DUSTY_MATRIX_MIRROR) != 0;
  const int compact_rows = (flags & DUSTY_MATRIX_COMPACT_ROWS) != 0, prepared = (flags & DUSTY_MATRIX_PREPARED) != 0;
  const int merge = (flags & DUSTY_MATRIX_MERGE_ORIGIN) != 0;
  if (mirror && (!symmetric || compact_rows)) return fail_arg(DUSTY_EINVAL, "chamfer_matrix: MIRROR needs SYMMETRIC and excludes COMPACT_ROWS");
  if (na < 0 || nb < 0 || pa <= 0 || pb <= 0) return fail_arg(DUSTY_EINVAL, "chamfer_matrix: bad sizes na=%d pa=%d nb=%d pb=%d", na, pa, nb, pb);
  if (symmetric && (nb != na || pb != pa)) return fail_arg(DUSTY_EINVAL, "chamfer_matrix: symmetric needs nb==na and pb==pa");
  if (row_stride <= 0 || row_begin < 0 || row_end > na || (M && ldm < nb))
    return fail_arg(DUSTY_EINVAL, "chamfer_matrix: bad row range [%d,%d) stride %d of %d, ldm %lld", row_begin, row_end, row_stride, na, ldm);
  if (fk.keys && (fk.n_ref < 0 || fk.off_a < 0 || fk.off_b < 0 || fk.off_a + na > fk.n_total || fk.off_b + nb > fk.n_total ||
                  (symmetric && fk.off_a != fk.off_b)))
    return fail_arg(DUSTY_EINVAL, "chamfer_matrix_fused: offsets %d+%d, %d+%d do not fit %d stacked clouds", fk.off_a, na, fk.off_b, nb, fk.n_total);
  if (row_begin >= row_end || nb == 0) return 0;
  if (int rc = check_device()) return rc;
  if (!A || !B || (!M && !fk.keys) || !workspace) return fail_arg(DUSTY_EINVAL, "chamfer_matrix: null pointer");
  if (!aligned16(workspace)) return fail_arg(DUSTY_EALIGN, "chamfer_matrix: workspace must be 16-byte aligned");
  const size_t need = dusty_chamfer_matrix_workspace_bytes(na, pa, symmetric ? 0 : nb, pb);
  if (workspace_bytes < need) return fail_arg(DUSTY_ENOSPACE, "chamfer_matrix: workspace %zu < %zu", workspace_bytes, need);
  // workspace: [scan A][meta A][boxes A]([scan B][meta B][boxes B])
  char* const wsp = static_cast<char*>(workspace);
  float4* sa = reinterpret_cast<float4*>(wsp);
  int2* ma = reinterpret_cast<int2*>(wsp + align_up(scan_bytes(na, pa), 256));
  float4* ba = reinterpret_cast<float4*>(wsp + align_up(scan_bytes(na, pa), 256) + meta_bytes(na));
  char* const wsb = wsp + align_up(scan_bytes(na, pa), 256) + meta_bytes(na) + box_bytes(na, pa);
  float4* sb = symmetric ? sa : reinterpret_cast<float4*>(wsb);
  int2* mb = symmetric ? ma : reinterpret_cast<int2*>(wsb + align_up(scan_bytes(nb, pb), 256));
  float4* bb = symmetric ? ba : reinterpret_cast<float4*>(wsb + align_up(scan_bytes(nb, pb), 256) + meta_bytes(nb));
  // Merged clouds that fit the shared-memory sort are put in k-d order with a box per chunk and per block of 32 chunks.
  // Clouds that fit shared memory twice over (the evaluation's 2048 FPS samples) go to the resident-pair kernel, larger
  // sorted ones to the two-level best-first walk from global memory, merged clouds beyond SORT_CAP to nn_kernel.
  const bool pair = merge && pa <= PAIR_CAP && pb <= PAIR_CAP;
  const bool walk = merge && !pair && pa <= SORT_CAP && pb <= SORT_CAP;
  const bool sorted = pair || walk;
  if (!prepared) {
    if (sorted) {
      if (int rc = run_prep_sort2(sort_side(A, na, pa, sa, ma, ba, nullptr, nullptr), na,
                                  sort_side(B, nb, pb, sb, mb, bb, nullptr, nullptr), symmetric ? 0 : nb, st, true)) return rc;
    } else if (merge) {
      if (int rc = run_prep_merge(A, na, pa, sa, ma, st)) return rc;
      if (!symmetric) if (int rc = run_prep_merge(B, nb, pb, sb, mb, st)) return rc;
    } else {
      if (int rc = run_prep(A, na, pa, sa, st)) return rc;
      if (!symmetric) if (int rc = run_prep(B, nb, pb, sb, st)) return rc;
    }
  }
  const int rows = (row_end - row_begin + row_stride - 1) / row_stride;
  if (rows > 65535) return fail_arg(DUSTY_EINVAL, "chamfer_matrix: %d rows in one call exceeds 65535", rows);
  Params p{};
  p.scanX = sa; p.scanY = sb;
  p.countX = pa; p.countY = pb;
  p.paddedX = padded_of(pa); p.paddedY = padded_of(pb);
  p.strideX = p.paddedX; p.strideY = p.paddedY;
  p.row_begin = row_begin; p.row_stride = row_stride;
  p.symmetric = symmetric; p.mirror = mirror; p.compact_rows = compact_rows;
  p.M = M; p.ldm = ldm;
  p.keys = fk.keys; p.n_total = fk.n_total; p.n_ref = fk.n_ref; p.offX = fk.off_a; p.offY = fk.off_b;
  p.visited = g_visited_counter;
  const dim3 grid(nb, rows, 1);
  if (merge) {
    p.metaX = ma; p.metaY = mb;
    if (sorted) { p.boxX = ba; p.boxY = bb; p.bbX = block_boxes_of(ba, na, pa); p.bbY = symmetric ? p.bbX : block_boxes_of(bb, nb, pb); }
    if (pair) return launch_pair_split(p, grid, st);
    if (walk) return launch_walk_split<true>(p, grid, st);
    return launch_nn<8, true, true>(p, grid, st);
  }
  return dispatch_matrix(pa > pb ? pa : pb, p, grid, st);
}

extern "C" int dusty_chamfer_matrix(const float* A, int na, int pa, const float* B, int nb, int pb, int row_begin,
                                    int row_end, int row_stride, int flags, float* M, long long ldm, void* workspace,
                                    size_t workspace_bytes, void* stream) {
  if (!M) return fail_arg(DUSTY_EINVAL, "chamfer_matrix: null pointer");
  return matrix_impl(A, na, pa, B, nb, pb, row_begin, row_end, row_stride, flags, M, ldm, FusedKeys{}, workspace,
                     workspace_bytes, stream);
}

extern "C" size_t dusty_nn_keys_bytes(int n_total) { return n_total > 0 ? (size_t)3 * n_total * sizeof(unsigned long long) : 0; }

extern "C" int dusty_nn_keys_reset(uint64_t* keys, int n_total, void* stream) {
  if (n_total <= 0) return 0;
  if (!keys) return fail_arg(DUSTY_EINVAL, "nn_keys_reset: null pointer");
  DUSTY_CUDA(cudaMemsetAsync(keys, 0xff, dusty_nn_keys_bytes(n_total), static_cast<cudaStream_t>(stream)));
  return 0;
}

extern "C" int dusty_chamfer_matrix_fused(const float* A, int na, int pa, const float* B, int nb, int pb, int row_begin,
                                          int row_end, int row_stride, int flags, float* M, long long ldm, int stacked_offset_a,
                                          int stacked_offset_b, int n_ref, int n_total, uint64_t* keys, void* workspace,
                                          size_t workspace_bytes, void* stream) {
  if (!keys) return fail_arg(DUSTY_EINVAL, "chamfer_matrix_fused: null keys");
  FusedKeys fk;
  fk.keys = reinterpret_cast<unsigned long long*>(keys);
  fk.n_total = n_total; fk.n_ref = n_ref; fk.off_a = stacked_offset_a; fk.off_b = stacked_offset_b;
  return matrix_impl(A, na, pa, B, nb, pb, row_begin, row_end, row_stride, flags, M, ldm, fk, workspace, workspace_bytes, stream);
}

extern "C" int dusty_chamfer_count_pairs(int enable, uint64_t* pairs_out) {
  if (pairs_out) {
    *pairs_out = 0;
    if (g_visited_counter) {
      DUSTY_CUDA(cudaDeviceSynchronize());
      unsigned long long v = 0;
      DUSTY_CUDA(cudaMemcpy(&v, g_visited_counter, sizeof(v), cudaMemcpyDeviceToHost));
      *pairs_out = v;
    }
  }
  if (enable && !g_visited_counter) {
    DUSTY_CUDA(cudaMalloc(&g_visited_counter, sizeof(unsigned long long)));
  }
  if (g_visited_counter) DUSTY_CUDA(cudaMemset(g_visited_counter, 0, sizeof(unsigned long long)));
  if (!enable && g_visited_counter) { DUSTY_CUDA(cudaFree(g_visited_counter)); g_visited_counter = nullptr; }
  return 0;
}
