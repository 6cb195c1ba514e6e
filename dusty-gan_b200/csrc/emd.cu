// Approximate Earth Mover's Distance (the PSGN approxmatch of Fan et al. 2017 that the reference ships as
// utils/metrics/distance/emd/: approxmatch, matchcost, matchcostgrad1, matchcostgrad2).
//
// The reference keeps a dense (b, m, n) match matrix in global memory and read-modify-writes it ten times per
// pair. Here no match matrix exists. approxmatch records, per temperature level, the two factor vectors ratioL
// (n) and ratioR (m) -- 10 (n + m) floats per pair -- and every consumer rebuilds
//   match[l][k] = 0 + w_7 + w_6 + ... + w_-2,   w_j = __expf(level_j d2(k,l)) * ratioL_j[k] * ratioR_j[l]
// on the fly in the reference's order of operations. Every sum of the reference is sequential per row or per
// column (and its match update is the same contracted multiply-add as ours), so the cost comes out bit-equal to
// the reference kernels' while the state per 2048^2 pair drops from 16 MB to 160 KB. The price is ten extra
// ex2 per point pair in the cost pass.
//
// One CTA of 512 threads works on one cloud pair at a time (the matchcost reduction is defined over 512
// threads: thread t owns rows t, t+512, ...). The other cloud of each sweep is staged through shared memory in
// tiles; a cloud of at most PTS_CAP points stays resident for the whole sweep, larger ones stream. The
// remain/ratio vectors live in a per-CTA slice of the workspace (L2-resident). Grids are persistent: at most
// kSlots CTAs loop over the pairs, so the workspace does not grow with the number of pairs.
//
// Arithmetic is written as the reference writes it (same expressions, same contraction by nvcc), with __expf and
// the default -prec-div / -prec-sqrt; tests/test_gpu_emd.py checks bit-equality against oracle/emd_reference.cu.
#include "common.cuh"

namespace dusty {
namespace emd {

constexpr int TPB = 512;
constexpr int LEVELS = 10;                 // j = 7, 6, ..., -2
constexpr int PTS_CAP = 2048;              // points of the swept cloud per shared-memory tile
constexpr int RR_CAP = 1024;               // points per tile when the ten per-level factors come along
constexpr int kCtasPerSM = 2;
constexpr int kSlots = kNumSMs * kCtasPerSM;
constexpr size_t kSmemBytes = sizeof(float4) * PTS_CAP + sizeof(float) * LEVELS * RR_CAP;

// per-pair state in the workspace slice of one CTA: remainL (n), remainR (m), then (if the caller keeps no
// factors) the factors (LEVELS, n + m): level index v = 7 - j holds ratioL_j (n) then ratioR_j (m)
__host__ __device__ inline size_t slot_floats(int n, int m) { return (size_t)(2 + LEVELS) * ((size_t)n + m); }
inline size_t slot_bytes(int n, int m) { return align_up(sizeof(float) * slot_floats(n, m), 256); }

__device__ __forceinline__ float level_of(int v) {     // level of index v = 7 - j, exactly as the reference forms it
  const int j = 7 - v;
  float level = -powf(4.0f, j);
  if (j == -2) level = 0;
  return level;
}

// One pass of approxmatch over the points of `own` (count n_own, one per thread and row group), summing over
// the points of `other` (count n_other, staged with weights w_other):
//   MODE 0 (pass 1, rows k):    s = 1e-9 + sum_l e * remainR[l];              ratioL[k] = remainL[k] / s
//   MODE 1 (pass 2, columns l): s = sum_k e * ratioL[k];                     ratioR, remainR update
//   MODE 2 (pass 3, rows k):    s = sum_l (e * ratioL[k]) * ratioR[l];        remainL[k] -= s (clamped at 0)
template <int MODE>
__device__ __forceinline__ void sweep(const float* __restrict__ own, int n_own, const float* __restrict__ other, int n_other,
                                      const float* w_other, float level, float* remain_own, float* ratio_own_in,
                                      float* ratio_own_out, float4* pts) {
  const int groups = (n_own + TPB - 1) / TPB;
  const bool resident = n_other <= PTS_CAP;
  for (int g = 0; g < groups; ++g) {
    const int k = g * TPB + threadIdx.x;
    float x1 = 0, y1 = 0, z1 = 0, rl = 0;
    if (k < n_own) {
      x1 = own[3 * k]; y1 = own[3 * k + 1]; z1 = own[3 * k + 2];
      if (MODE == 2) rl = ratio_own_in[k];
    }
    float s = MODE == 0 ? 1e-9f : 0.0f;
    for (int l0 = 0; l0 < n_other; l0 += PTS_CAP) {
      const int lend = min(n_other - l0, PTS_CAP);
      if (!resident || g == 0) {
        __syncthreads();
        for (int l = threadIdx.x; l < lend; l += TPB)
          pts[l] = make_float4(other[3 * (l0 + l)], other[3 * (l0 + l) + 1], other[3 * (l0 + l) + 2], w_other[l0 + l]);
        __syncthreads();
      }
      if (k < n_own) {
#pragma unroll 4
        for (int l = 0; l < lend; ++l) {
          const float4 q = pts[l];
          const float x2 = q.x, y2 = q.y, z2 = q.z;
          if (MODE == 2) s += __expf(level * ((x2 - x1) * (x2 - x1) + (y2 - y1) * (y2 - y1) + (z2 - z1) * (z2 - z1))) * rl * q.w;
          else s += __expf(level * ((x2 - x1) * (x2 - x1) + (y2 - y1) * (y2 - y1) + (z2 - z1) * (z2 - z1))) * q.w;
        }
      }
    }
    if (k < n_own) {
      if (MODE == 0) {
        ratio_own_out[k] = remain_own[k] / s;
      } else if (MODE == 1) {
        const float r = remain_own[k];
        s *= r;
        const float consumption = fminf(r / (s + 1e-9f), 1.0f);
        ratio_own_out[k] = consumption * r;
        remain_own[k] = fmaxf(0.0f, r - s);
      } else {
        remain_own[k] = fmaxf(0.0f, remain_own[k] - s);
      }
    }
  }
}

// approxmatch for one pair: fills fac (LEVELS, n + m). Ends with a barrier, so fac is visible to the CTA.
__device__ void approxmatch(const float* __restrict__ p1, const float* __restrict__ p2, int n, int m, float* remL,
                            float* remR, float* fac, float4* pts) {
  float multiL, multiR;
  if (n >= m) { multiL = 1; multiR = n / m; } else { multiL = m / n; multiR = 1; }
  for (int k = threadIdx.x; k < n; k += TPB) remL[k] = multiL;
  for (int l = threadIdx.x; l < m; l += TPB) remR[l] = multiR;
  for (int v = 0; v < LEVELS; ++v) {
    const float level = level_of(v);
    float* ratioL = fac + (size_t)v * (n + m);
    float* ratioR = ratioL + n;
    sweep<0>(p1, n, p2, m, remR, level, remL, nullptr, ratioL, pts);
    sweep<1>(p2, m, p1, n, ratioL, level, remR, nullptr, ratioR, pts);
    sweep<2>(p1, n, p2, m, ratioR, level, remL, ratioL, nullptr, pts);
  }
  __syncthreads();
}

// Per-pair consumers of the rebuilt match. Thread t owns the points t, t+512, ... of `own`; for each it walks
// the points of `other` in order, staged in tiles of RR_CAP with their ten factors.
//   COST: own = cloud 1 rows k, returns this thread's matchcost running sum (before the tree).
//   GRAD: gradient of the owned point (d cost / d own, unscaled), as matchcostgrad1 / 2 form it.
// `own_fac` / `other_fac` point at the level-0 factor of each cloud (stride n + m between levels).
template <bool GRAD>
__device__ __forceinline__ float walk(const float* __restrict__ own, int n_own, const float* own_fac,
                                      const float* __restrict__ other, int n_other, const float* other_fac,
                                      int stride, bool own_is_1, float4* pts, float* rrs, float* grad_out, float scale) {
  float lv[LEVELS];
#pragma unroll
  for (int v = 0; v < LEVELS; ++v) lv[v] = level_of(v);
  float subsum = 0;
  const int groups = (n_own + TPB - 1) / TPB;
  const bool resident = n_other <= RR_CAP;
  for (int g = 0; g < groups; ++g) {
    const int k = g * TPB + threadIdx.x;
    float x1 = 0, y1 = 0, z1 = 0, fo[LEVELS];
#pragma unroll
    for (int v = 0; v < LEVELS; ++v) fo[v] = 0;
    if (k < n_own) {
      x1 = own[3 * k]; y1 = own[3 * k + 1]; z1 = own[3 * k + 2];
#pragma unroll
      for (int v = 0; v < LEVELS; ++v) fo[v] = own_fac[(size_t)v * stride + k];
    }
    float gx = 0, gy = 0, gz = 0;
    for (int l0 = 0; l0 < n_other; l0 += RR_CAP) {
      const int lend = min(n_other - l0, RR_CAP);
      if (!resident || g == 0) {
        __syncthreads();
        for (int l = threadIdx.x; l < lend; l += TPB) {
          pts[l] = make_float4(other[3 * (l0 + l)], other[3 * (l0 + l) + 1], other[3 * (l0 + l) + 2], 0.0f);
#pragma unroll
          for (int v = 0; v < LEVELS; ++v) rrs[v * RR_CAP + l] = other_fac[(size_t)v * stride + l0 + l];
        }
        __syncthreads();
      }
      if (k < n_own) {
#pragma unroll 1
        for (int l = 0; l < lend; ++l) {
          const float4 q = pts[l];
          const float x2 = q.x, y2 = q.y, z2 = q.z;
          const float d2 = (x2 - x1) * (x2 - x1) + (y2 - y1) * (y2 - y1) + (z2 - z1) * (z2 - z1);
          float match = 0;
          // w = (e * ratioL) * ratioR: the factor of cloud 1 multiplies first
#pragma unroll
          for (int v = 0; v < LEVELS; ++v) {
            if (own_is_1) match += __expf(lv[v] * d2) * fo[v] * rrs[v * RR_CAP + l];
            else match += __expf(lv[v] * d2) * rrs[v * RR_CAP + l] * fo[v];
          }
          if (GRAD) {
            const float d = fmaxf(sqrtf(d2), 1e-20f);
            const float c = match / d;
            gx += (x1 - x2) * c; gy += (y1 - y2) * c; gz += (z1 - z2) * c;
          } else {
            subsum += sqrtf(d2) * match;
          }
        }
      }
    }
    if (GRAD && k < n_own) {
      grad_out[3 * k] = gx * scale; grad_out[3 * k + 1] = gy * scale; grad_out[3 * k + 2] = gz * scale;
    }
  }
  return subsum;
}

// matchcost's tree: allsum[t] += allsum[t + s] for s = 1, 2, 4, ... where (t & s) == 0
__device__ __forceinline__ float tree_sum(float subsum, float* allsum) {
  allsum[threadIdx.x] = subsum;
  for (int s = 1; s < TPB; s <<= 1) {
    __syncthreads();
    if ((threadIdx.x & s) == 0 && threadIdx.x + s < TPB) allsum[threadIdx.x] += allsum[threadIdx.x + s];
  }
  __syncthreads();
  const float r = allsum[0];
  __syncthreads();
  return r;
}

__device__ __forceinline__ float pair_cost(const float* p1, const float* p2, int n, int m, float* remL, float* remR,
                                           float* fac, float4* pts, float* rrs, float* allsum) {
  approxmatch(p1, p2, n, m, remL, remR, fac, pts);
  const float sub = walk<false>(p1, n, fac, p2, m, fac + n, n + m, true, pts, rrs, nullptr, 0.0f);
  return tree_sum(sub, allsum);
}

__global__ void __launch_bounds__(TPB, kCtasPerSM) emd_forward_kernel(const float* __restrict__ xyz1,
                                                                      const float* __restrict__ xyz2, int b, int n, int m,
                                                                      float* __restrict__ cost, float* factors,
                                                                      float* ws, size_t slot_stride) {
  extern __shared__ float4 smem[];
  __shared__ float allsum[TPB];
  float4* pts = smem;
  float* rrs = reinterpret_cast<float*>(smem + PTS_CAP);
  float* remL = ws + blockIdx.x * slot_stride;
  float* remR = remL + n;
  for (int i = blockIdx.x; i < b; i += gridDim.x) {
    float* fac = factors ? factors + (size_t)i * LEVELS * (n + m) : remR + m;
    const float c = pair_cost(xyz1 + (size_t)i * n * 3, xyz2 + (size_t)i * m * 3, n, m, remL, remR, fac, pts, rrs, allsum);
    if (threadIdx.x == 0) cost[i] = c;
  }
}

// grad1 rows (blockIdx.y == 0) or grad2 columns (blockIdx.y == 1) of every pair, from the saved factors
__global__ void __launch_bounds__(TPB, kCtasPerSM) emd_backward_kernel(const float* __restrict__ xyz1,
                                                                       const float* __restrict__ xyz2, int b, int n, int m,
                                                                       const float* __restrict__ grad_cost,
                                                                       const float* __restrict__ factors,
                                                                       float* __restrict__ grad1, float* __restrict__ grad2) {
  extern __shared__ float4 smem[];
  float4* pts = smem;
  float* rrs = reinterpret_cast<float*>(smem + PTS_CAP);
  for (int i = blockIdx.x; i < b; i += gridDim.x) {
    const float* p1 = xyz1 + (size_t)i * n * 3;
    const float* p2 = xyz2 + (size_t)i * m * 3;
    const float* fac = factors + (size_t)i * LEVELS * (n + m);
    const float g = grad_cost[i];
    if (blockIdx.y == 0) walk<true>(p1, n, fac, p2, m, fac + n, n + m, true, pts, rrs, grad1 + (size_t)i * n * 3, g);
    else walk<true>(p2, m, fac + n, p1, n, fac, n + m, false, pts, rrs, grad2 + (size_t)i * m * 3, g);
  }
}

struct MatrixArgs {
  const float* A; int na, pa;
  const float* B; int nb, pb;
  int row_begin, row_stride, rows;
  float* M; long long ldm;
  float inv_pa;                              // f32(1 / pa): compute_emd divides the cost by the point count
  unsigned long long* keys; int off_a, off_b, n_ref, n_total;
  float* ws; size_t slot_stride;
};

__global__ void __launch_bounds__(TPB, kCtasPerSM) emd_matrix_kernel(const MatrixArgs p) {
  extern __shared__ float4 smem[];
  __shared__ float allsum[TPB];
  float4* pts = smem;
  float* rrs = reinterpret_cast<float*>(smem + PTS_CAP);
  float* remL = p.ws + blockIdx.x * p.slot_stride;
  float* remR = remL + p.pa;
  float* fac = remR + p.pb;
  const long long entries = (long long)p.rows * p.nb;
  for (long long e = blockIdx.x; e < entries; e += gridDim.x) {
    const int i = p.row_begin + (int)(e / p.nb) * p.row_stride, j = (int)(e % p.nb);
    const float c = pair_cost(p.A + (size_t)i * p.pa * 3, p.B + (size_t)j * p.pb * 3, p.pa, p.pb, remL, remR, fac, pts,
                              rrs, allsum);
    if (threadIdx.x == 0) {
      const float v = c * p.inv_pa;
      if (p.M) p.M[(long long)i * p.ldm + j] = v;
      // packed (value bits << 32 | stacked index) minima as in the Chamfer matrix epilogue (v >= 0). The 1-NN
      // matrix [[M_rr, M_rg], [M_rg^T, M_gg]] is reduced column-wise: entry (r, c) feeds column c; an M_rg entry
      // also stands at (c, r) and feeds both cross-set minima.
      if (p.keys) {
        const int r = p.off_a + i, col = p.off_b + j;
        const unsigned long long vb = (unsigned long long)__float_as_uint(v) << 32;
        if (r != col) atomicMin(p.keys + col, vb | (unsigned)r);
        if (r < p.n_ref && col >= p.n_ref) {
          atomicMin(p.keys + r, vb | (unsigned)col);
          atomicMin(p.keys + p.n_total + col, vb | (unsigned)r);
          atomicMin(p.keys + 2 * (long long)p.n_total + r, vb | (unsigned)col);
        }
      }
    }
  }
}

template <typename K>
int set_smem(K kernel) {
  static bool done[kMaxDevices] = {};
  const int dev = current_device();
  if (!done[dev]) {
    DUSTY_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemBytes));
    done[dev] = true;
  }
  return 0;
}

}  // namespace emd
}  // namespace dusty

using namespace dusty;
using namespace dusty::emd;

extern "C" size_t dusty_emd_forward_workspace_bytes(int b, int n, int m) {
  if (b <= 0 || n <= 0 || m <= 0) return 0;
  return (size_t)(b < kSlots ? b : kSlots) * slot_bytes(n, m);
}

extern "C" int dusty_emd_forward(const float* xyz1, const float* xyz2, int b, int n, int m, float* cost, float* factors,
                                 void* ws, size_t ws_bytes, void* stream) {
  if (b < 0 || n <= 0 || m <= 0) return fail_arg(DUSTY_EINVAL, "emd_forward: bad sizes b=%d n=%d m=%d (clouds must hold points)", b, n, m);
  if (b == 0) return 0;
  if (int rc = check_device()) return rc;
  if (!xyz1 || !xyz2 || !cost || !ws) return fail_arg(DUSTY_EINVAL, "emd_forward: null pointer");
  const size_t need = dusty_emd_forward_workspace_bytes(b, n, m);
  if (ws_bytes < need) return fail_arg(DUSTY_ENOSPACE, "emd_forward: workspace %zu < %zu", ws_bytes, need);
  if (int rc = set_smem(emd_forward_kernel)) return rc;
  const int grid = b < kSlots ? b : kSlots;
  emd_forward_kernel<<<grid, TPB, kSmemBytes, static_cast<cudaStream_t>(stream)>>>(
      xyz1, xyz2, b, n, m, cost, factors, static_cast<float*>(ws), slot_bytes(n, m) / sizeof(float));
  DUSTY_AFTER_LAUNCH("emd_forward_kernel");
  return 0;
}

extern "C" int dusty_emd_backward(const float* xyz1, const float* xyz2, int b, int n, int m, const float* grad_cost,
                                  const float* factors, float* grad1, float* grad2, void* ws, size_t ws_bytes, void* stream) {
  (void)ws; (void)ws_bytes;       // no scratch: the match is rebuilt from the factors
  if (b < 0 || n <= 0 || m <= 0) return fail_arg(DUSTY_EINVAL, "emd_backward: bad sizes b=%d n=%d m=%d (clouds must hold points)", b, n, m);
  if (b == 0) return 0;
  if (int rc = check_device()) return rc;
  if (!xyz1 || !xyz2 || !grad_cost || !factors || !grad1 || !grad2) return fail_arg(DUSTY_EINVAL, "emd_backward: null pointer");
  if (int rc = set_smem(emd_backward_kernel)) return rc;
  const int grid = b < kSlots / 2 ? b : kSlots / 2;
  emd_backward_kernel<<<dim3(grid, 2), TPB, kSmemBytes, static_cast<cudaStream_t>(stream)>>>(xyz1, xyz2, b, n, m, grad_cost,
                                                                                            factors, grad1, grad2);
  DUSTY_AFTER_LAUNCH("emd_backward_kernel");
  return 0;
}

extern "C" size_t dusty_emd_matrix_workspace_bytes(int na, int pa, int nb, int pb) {
  if (na <= 0 || nb <= 0 || pa <= 0 || pb <= 0) return 0;
  return (size_t)kSlots * slot_bytes(pa, pb);
}

extern "C" int dusty_emd_matrix(const float* A, int na, int pa, const float* B, int nb, int pb, int row_begin, int row_end,
                                int row_stride, float* M, long long ldm, int stacked_offset_a, int stacked_offset_b,
                                int n_ref, int n_total, uint64_t* keys, void* ws, size_t ws_bytes, void* stream) {
  if (na < 0 || nb < 0 || pa <= 0 || pb <= 0)
    return fail_arg(DUSTY_EINVAL, "emd_matrix: bad sizes na=%d pa=%d nb=%d pb=%d (clouds must hold points)", na, pa, nb, pb);
  if (row_stride <= 0 || row_begin < 0 || row_end > na || (M && ldm < nb))
    return fail_arg(DUSTY_EINVAL, "emd_matrix: bad row range [%d,%d) stride %d of %d, ldm %lld", row_begin, row_end, row_stride, na, ldm);
  if (keys) {
    const int a0 = stacked_offset_a, a1 = stacked_offset_a + na, b0 = stacked_offset_b, b1 = stacked_offset_b + nb;
    if (n_ref < 0 || a0 < 0 || b0 < 0 || a1 > n_total || b1 > n_total)
      return fail_arg(DUSTY_EINVAL, "emd_matrix: offsets %d+%d, %d+%d do not fit %d stacked clouds", a0, na, b0, nb, n_total);
    const bool a_ref = a1 <= n_ref, a_gen = a0 >= n_ref, b_ref = b1 <= n_ref, b_gen = b0 >= n_ref;
    if (!(a_ref || a_gen) || !(b_ref || b_gen))
      return fail_arg(DUSTY_EINVAL, "emd_matrix: a set straddles the reference/generated boundary %d", n_ref);
    if (a_gen && b_ref && !(a_ref || b_gen))
      return fail_arg(DUSTY_EINVAL, "emd_matrix: generated-by-reference launch (M_gr is never part of the scores)");
  }
  if (row_begin >= row_end || nb == 0) return 0;
  if (int rc = check_device()) return rc;
  if (!A || !B || (!M && !keys) || !ws) return fail_arg(DUSTY_EINVAL, "emd_matrix: null pointer");
  const size_t need = dusty_emd_matrix_workspace_bytes(na, pa, nb, pb);
  if (ws_bytes < need) return fail_arg(DUSTY_ENOSPACE, "emd_matrix: workspace %zu < %zu", ws_bytes, need);
  if (int rc = set_smem(emd_matrix_kernel)) return rc;
  MatrixArgs p{};
  p.A = A; p.na = na; p.pa = pa; p.B = B; p.nb = nb; p.pb = pb;
  p.row_begin = row_begin; p.row_stride = row_stride; p.rows = (row_end - row_begin + row_stride - 1) / row_stride;
  p.M = M; p.ldm = ldm;
  p.inv_pa = (float)(1.0 / (double)pa);
  p.keys = reinterpret_cast<unsigned long long*>(keys); p.off_a = stacked_offset_a; p.off_b = stacked_offset_b;
  p.n_ref = n_ref; p.n_total = n_total;
  p.ws = static_cast<float*>(ws); p.slot_stride = slot_bytes(pa, pb) / sizeof(float);
  const long long entries = (long long)p.rows * nb;
  const int grid = entries < kSlots ? (int)entries : kSlots;
  emd_matrix_kernel<<<grid, TPB, kSmemBytes, static_cast<cudaStream_t>(stream)>>>(p);
  DUSTY_AFTER_LAUNCH("emd_matrix_kernel");
  return 0;
}
