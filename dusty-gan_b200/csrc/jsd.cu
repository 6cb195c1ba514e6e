// Jensen-Shannon divergence between occupancy histograms (SURVEY.md 8f-2) for sm_100a.
//
// Replaces entropy_of_occupancy_grid's voting (reference utils/metrics/jsd.py:23-92): a brute-force
// arg-min of every point against every in-sphere point of a resolution^3 grid (10 144 candidates at
// 28^3 -> 2.1e11 distance evaluations for two sets of 5000 clouds of 2048 points), done there in three
// nested Python loops.
// On a regular grid the nearest candidate is found from the point's own cell:
//   * the 5x5x5 neighbourhood of the rounded cell is searched with the reference's arithmetic
//     (f32 differences, squares, (dx^2 + dy^2) + dz^2, lowest grid index on ties);
//   * every grid point outside that neighbourhood is at least 2.5 spacings away, so the result is
//     the global arg-min whenever the best distance is below (2.4 spacing)^2; otherwise (points
//     well outside the sphere) the kernel falls back to the full scan the reference does.
// One CTA per cloud keeps the cloud's histogram in shared memory, which gives both outputs of the
// reference at once: counters (points per cell) and the per-cell number of clouds that touch it.
#include "common.cuh"

namespace dusty {
namespace jsd {

constexpr int TPB = 256;

__device__ __forceinline__ float dist_ref(float px, float py, float pz, const float* g) {
  const float dx = __fsub_rn(px, g[0]), dy = __fsub_rn(py, g[1]), dz = __fsub_rn(pz, g[2]);
  return __fadd_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), __fmul_rn(dz, dz));
}

// grid (ng,3): the in-sphere grid points in the reference's order; cell_to_idx (res^3): compact
// index of a cell or -1; axis (res): the grid coordinates along one axis.
__global__ void __launch_bounds__(TPB) vote_kernel(const float* __restrict__ pcs, int npts, int res, int ng,
                                                   const float* __restrict__ grid, const int* __restrict__ cell_to_idx,
                                                   const float* __restrict__ axis, float spacing,
                                                   unsigned* __restrict__ counters, unsigned* __restrict__ clouds_touching) {
  extern __shared__ unsigned hist[];      // ng counters of this cloud
  for (int c = threadIdx.x; c < ng; c += TPB) hist[c] = 0u;
  __syncthreads();
  const float* cloud = pcs + (long long)blockIdx.x * npts * 3;
  const float inv_spacing = 1.0f / spacing;
  const float safe = (2.4f * spacing) * (2.4f * spacing);
  for (int p = threadIdx.x; p < npts; p += TPB) {
    const float px = cloud[3 * p], py = cloud[3 * p + 1], pz = cloud[3 * p + 2];
    const int cx = min(res - 1, max(0, __float2int_rn((px + 0.5f) * inv_spacing)));
    const int cy = min(res - 1, max(0, __float2int_rn((py + 0.5f) * inv_spacing)));
    const int cz = min(res - 1, max(0, __float2int_rn((pz + 0.5f) * inv_spacing)));
    float best = __int_as_float(0x7f800000);
    int bi = 0x7fffffff;
    for (int ix = max(0, cx - 2); ix <= min(res - 1, cx + 2); ++ix)
      for (int iy = max(0, cy - 2); iy <= min(res - 1, cy + 2); ++iy)
        for (int iz = max(0, cz - 2); iz <= min(res - 1, cz + 2); ++iz) {
          const int id = cell_to_idx[(ix * res + iy) * res + iz];
          if (id < 0) continue;
          const float g[3] = {axis[ix], axis[iy], axis[iz]};
          const float d = dist_ref(px, py, pz, g);
          if (d < best || (d == best && id < bi)) { best = d; bi = id; }
        }
    if (!(best < safe)) {                 // far from every in-sphere cell (or NaN): the reference's full scan
      best = __int_as_float(0x7f800000);
      bi = 0;
      for (int id = 0; id < ng; ++id) {
        const float d = dist_ref(px, py, pz, grid + 3 * id);
        if (id == 0 || d < best) { best = d; bi = id; }
      }
    }
    atomicAdd(&hist[bi], 1u);
  }
  __syncthreads();
  for (int c = threadIdx.x; c < ng; c += TPB) {
    const unsigned h = hist[c];
    if (h) { atomicAdd(&counters[c], h); atomicAdd(&clouds_touching[c], 1u); }
  }
}

__device__ __forceinline__ double block_sum(double v, double* sm) {
  #pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = v;
  __syncthreads();
  double s = 0.0;
  #pragma unroll
  for (int w = 0; w < TPB / 32; ++w) s += sm[w];
  return s;
}

// _jensen_shannon_divergence (reference jsd.py:110-121) with _entropy's in-place "p += eps"
// (jsd.py:95-107): e1 = H2(P_+eps), e2 = H2(Q_+eps), e_sum = H2(((P_+eps) + (Q_+eps)) / 2 + eps).
__global__ void __launch_bounds__(TPB) jsd_kernel(const unsigned* __restrict__ P, const unsigned* __restrict__ Q, int ng,
                                                  float* __restrict__ out) {
  __shared__ double sm[TPB / 32];
  double sp = 0, sq = 0;
  for (int c = threadIdx.x; c < ng; c += TPB) { sp += P[c]; sq += Q[c]; }
  const float fp = (float)block_sum(sp, sm), fq = (float)block_sum(sq, sm);   // counts are exact in f32 sums below 2^24
  const float eps = 1e-8f;
  double e1 = 0, e2 = 0, es = 0;
  for (int c = threadIdx.x; c < ng; c += TPB) {
    const float p = __fadd_rn(__fdiv_rn((float)P[c], fp), eps);
    const float q = __fadd_rn(__fdiv_rn((float)Q[c], fq), eps);
    const float m = __fadd_rn(__fmul_rn(__fadd_rn(p, q), 0.5f), eps);
    e1 += (double)__fmul_rn(-p, log2f(p));
    e2 += (double)__fmul_rn(-q, log2f(q));
    es += (double)__fmul_rn(-m, log2f(m));
  }
  e1 = block_sum(e1, sm); e2 = block_sum(e2, sm); es = block_sum(es, sm);
  if (threadIdx.x == 0) out[0] = (float)es - ((float)e1 + (float)e2) * 0.5f;
}

}  // namespace jsd
}  // namespace dusty

using namespace dusty;
using namespace dusty::jsd;

extern "C" int dusty_jsd_vote(const float* pcs, int b, int npts, int resolution, int ng, const float* grid,
                              const int32_t* cell_to_idx, const float* axis, float spacing, uint32_t* counters,
                              uint32_t* clouds_touching, void* stream) {
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (b < 0 || npts < 0 || resolution < 2 || ng <= 0) return fail_arg(DUSTY_EINVAL, "jsd_vote: bad sizes b=%d npts=%d res=%d ng=%d", b, npts, resolution, ng);
  if (ng > 48 * 1024) return fail_arg(DUSTY_EINVAL, "jsd_vote: %d grid points exceed the 48k shared-memory histogram", ng);
  if (!counters || !clouds_touching) return fail_arg(DUSTY_EINVAL, "jsd_vote: null pointer");
  if (int rc = check_device()) return rc;
  DUSTY_CUDA(cudaMemsetAsync(counters, 0, sizeof(uint32_t) * ng, st));
  DUSTY_CUDA(cudaMemsetAsync(clouds_touching, 0, sizeof(uint32_t) * ng, st));
  if (b == 0 || npts == 0) return 0;
  if (!pcs || !grid || !cell_to_idx || !axis) return fail_arg(DUSTY_EINVAL, "jsd_vote: null pointer");
  const size_t smem = sizeof(unsigned) * (size_t)ng;
  static size_t configured[kMaxDevices] = {};
  const int dev = current_device();
  if (smem > configured[dev]) {
    DUSTY_CUDA(cudaFuncSetAttribute(vote_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    configured[dev] = smem;
  }
  vote_kernel<<<b, TPB, smem, st>>>(pcs, npts, resolution, ng, grid, cell_to_idx, axis, spacing, counters, clouds_touching);
  DUSTY_AFTER_LAUNCH("jsd vote_kernel");
  return 0;
}

extern "C" int dusty_jsd_from_counts(const uint32_t* counts_p, const uint32_t* counts_q, int ng, float* out, void* stream) {
  if (ng <= 0 || !counts_p || !counts_q || !out) return fail_arg(DUSTY_EINVAL, "jsd_from_counts: bad arguments");
  if (int rc = check_device()) return rc;
  jsd_kernel<<<1, TPB, 0, static_cast<cudaStream_t>(stream)>>>(counts_p, counts_q, ng, out);
  DUSTY_AFTER_LAUNCH("jsd_kernel");
  return 0;
}
