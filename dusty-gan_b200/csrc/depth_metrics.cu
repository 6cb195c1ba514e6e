// Reconstruction metrics of range images (reference utils/metrics/depth.py, called by evaluate_reconstruction.py;
// the contract is restated in DESIGN.md §2.8) for sm_100a.
//
// Both images of a pair go through the reference's postprocess chain, rounded where ATen's element-wise kernels
// round it (the same operations as the first half of range_from_inv in head_project.cu):
//   inv   = clamp((x + 1) * 0.5, 0, 1)                 tanh_to_sigmoid + clamp_; NaN survives the clamp as in torch
//   valid = |inv| > tol
//   m     = (1 / (inv * disp_scale + disp_shift)) * valid        revert_depth(norm=False), metres
// and every pixel valid on both sides adds, in double from the two f32 depths p and t (d = p - t):
//   |d| * (1/t), d^2 * (1/t), d^2, (log p - log t)^2, and the three delta counts max(p/t, t/p) < 1.25^k,
// each tested as p < 1.25^k t && t < 1.25^k p: 1.25^k t is exact in double, and a quotient of two floats cannot round
// onto 1.25^k from below, so the counts equal those of the rounded quotients.
//
//   depth_chunk_kernel    one CTA per (image, chunk of 1024 pixels): two 128-bit loads per image and thread, the
//                         per-thread sums reduced over the warp (redux for counts, a fixed xor butterfly for doubles)
//                         and over the four warps in warp order -> (b, chunks, 10) partials in the workspace;
//   depth_combine_kernel  one thread per (image, sum): the chunk partials added in chunk order.
// The chunk count depends on h*w only and nothing is reduced with atomics, so a scan's sums are bit-identical from call
// to call and do not depend on the other scans of the batch.
#include "common.cuh"

namespace dusty {
namespace depth {

constexpr int TPB = 128;
constexpr int GROUPS = 2;                      // float4 groups per thread and image
constexpr int CHUNK = TPB * GROUPS * 4;        // pixels per CTA
constexpr int NSUM = 10;

__device__ __forceinline__ float metres(float x, const dusty_head_params& p, bool& valid) {
  float inv = __fmul_rn(__fadd_rn(x, 1.0f), 0.5f);
  inv = inv < 0.0f ? 0.0f : (inv > 1.0f ? 1.0f : inv);
  valid = fabsf(inv) > p.tol;
  const float depth = __frcp_rn(__fadd_rn(__fmul_rn(inv, p.disp_scale), p.disp_shift));   // == 1.0f / disp
  return __fmul_rn(depth, valid ? 1.0f : 0.0f);
}

struct Acc {
  double absrel = 0.0, sqrel = 0.0, sq = 0.0, lg = 0.0;
  unsigned both = 0, pv = 0, tv = 0, a1 = 0, a2 = 0, a3 = 0;
};

__device__ __forceinline__ void accumulate(float pm, bool vp, float tm, bool vt, Acc& a) {
  a.pv += vp;
  a.tv += vt;
  if (!(vp && vt)) return;
  const double P = pm, T = tm;
  const double d = P - T;
  const double rt = 1.0 / T;
  const double d2 = __dmul_rn(d, d);
  const double l = log(P) - log(T);
  a.both += 1;
  a.absrel += __dmul_rn(fabs(d), rt);
  a.sqrel += __dmul_rn(d2, rt);
  a.sq += d2;
  a.lg += __dmul_rn(l, l);
  a.a1 += (P < 1.25 * T && T < 1.25 * P);
  a.a2 += (P < 1.5625 * T && T < 1.5625 * P);
  a.a3 += (P < 1.953125 * T && T < 1.953125 * P);
}

__device__ __forceinline__ double warp_sum(double v) {
  #pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

__global__ void __launch_bounds__(TPB) depth_chunk_kernel(const dusty_head_params p, const float* __restrict__ pred,
                                                          const float* __restrict__ target, float* out_pred,
                                                          float* out_target, double* __restrict__ partial, int npix,
                                                          int chunks) {
  __shared__ double red[TPB / 32][NSUM];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const long long img = blockIdx.x / chunks;
  const int chunk = (int)(blockIdx.x - (unsigned)img * chunks);
  const long long base = img * npix;
  float4 pv[GROUPS], tv[GROUPS];
  int pix[GROUPS];
  #pragma unroll
  for (int g = 0; g < GROUPS; ++g) {
    pix[g] = chunk * CHUNK + (g * TPB + tid) * 4;
    if (pix[g] < npix) {
      pv[g] = ldg_stream(reinterpret_cast<const float4*>(pred + base + pix[g]));
      tv[g] = ldg_stream(reinterpret_cast<const float4*>(target + base + pix[g]));
    }
  }
  Acc a;
  #pragma unroll
  for (int g = 0; g < GROUPS; ++g) {
    if (pix[g] >= npix) continue;
    const float px[4] = {pv[g].x, pv[g].y, pv[g].z, pv[g].w};
    const float tx[4] = {tv[g].x, tv[g].y, tv[g].z, tv[g].w};
    float pm[4], tm[4];
    bool vp[4], vt[4];
    #pragma unroll
    for (int q = 0; q < 4; ++q) {
      pm[q] = metres(px[q], p, vp[q]);
      tm[q] = metres(tx[q], p, vt[q]);
    }
    if (out_pred) stg_stream(reinterpret_cast<float4*>(out_pred + base + pix[g]), make_float4(pm[0], pm[1], pm[2], pm[3]));
    if (out_target)
      stg_stream(reinterpret_cast<float4*>(out_target + base + pix[g]), make_float4(tm[0], tm[1], tm[2], tm[3]));
    #pragma unroll
    for (int q = 0; q < 4; ++q) accumulate(pm[q], vp[q], tm[q], vt[q], a);
  }
  const unsigned full = 0xffffffffu;
  const double w[NSUM] = {(double)__reduce_add_sync(full, a.both), (double)__reduce_add_sync(full, a.pv),
                          (double)__reduce_add_sync(full, a.tv), warp_sum(a.absrel), warp_sum(a.sqrel),
                          warp_sum(a.sq), warp_sum(a.lg), (double)__reduce_add_sync(full, a.a1),
                          (double)__reduce_add_sync(full, a.a2), (double)__reduce_add_sync(full, a.a3)};
  if (lane == 0) {
    #pragma unroll
    for (int k = 0; k < NSUM; ++k) red[warp][k] = w[k];
  }
  __syncthreads();
  if (tid < NSUM) {
    double s = red[0][tid];
    #pragma unroll
    for (int k = 1; k < TPB / 32; ++k) s += red[k][tid];
    partial[((long long)img * chunks + chunk) * NSUM + tid] = s;
  }
}

__global__ void __launch_bounds__(256) depth_combine_kernel(const double* __restrict__ partial, double* __restrict__ sums,
                                                            int b, int chunks) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)b * NSUM) return;
  const long long img = i / NSUM;
  const int k = (int)(i - img * NSUM);
  const double* q = partial + img * chunks * NSUM + k;
  double s = q[0];
  for (int c = 1; c < chunks; ++c) s += q[(long long)c * NSUM];
  sums[i] = s;
}

int chunks_of(int h, int w) { return (int)(((long long)h * w + CHUNK - 1) / CHUNK); }

int check_shape(int b, int h, int w) {
  if (b < 0 || h <= 0 || w <= 0) return fail_arg(DUSTY_EINVAL, "depth_metrics: bad shape b=%d h=%d w=%d", b, h, w);
  if (w % 4 != 0) return fail_arg(DUSTY_EINVAL, "depth_metrics: w=%d must be a multiple of 4", w);
  if ((long long)h * w > 0x7fffffffLL - CHUNK) return fail_arg(DUSTY_EINVAL, "depth_metrics: image too large");
  if ((long long)b * chunks_of(h, w) > 0x7fffffffLL)
    return fail_arg(DUSTY_EINVAL, "depth_metrics: %d images of %dx%d overflow the grid", b, h, w);
  return 0;
}

}  // namespace depth
}  // namespace dusty

using namespace dusty;
using namespace dusty::depth;

extern "C" size_t dusty_depth_metrics_workspace_bytes(int b, int h, int w) {
  if (b <= 0 || h <= 0 || w <= 0 || w % 4 != 0 || (long long)h * w > 0x7fffffffLL - CHUNK) return 0;
  return sizeof(double) * NSUM * (size_t)b * (size_t)chunks_of(h, w);
}

extern "C" int dusty_depth_metrics(const dusty_head_params* p, const float* pred, const float* target, double* sums,
                                   float* out_pred_m, float* out_target_m, void* workspace, size_t workspace_bytes,
                                   void* stream) {
  if (!p) return fail_arg(DUSTY_EINVAL, "depth_metrics: null params");
  if (int rc = check_shape(p->b, p->h, p->w)) return rc;
  if (p->b == 0) return 0;
  if (int rc = check_device()) return rc;
  if (!pred || !target || !sums || !workspace) return fail_arg(DUSTY_EINVAL, "depth_metrics: null pointer");
  if (!aligned16(pred) || !aligned16(target) || (out_pred_m && !aligned16(out_pred_m)) ||
      (out_target_m && !aligned16(out_target_m)))
    return fail_arg(DUSTY_EALIGN, "depth_metrics: images must be 16-byte aligned");
  if ((reinterpret_cast<uintptr_t>(sums) & 7u) || (reinterpret_cast<uintptr_t>(workspace) & 7u))
    return fail_arg(DUSTY_EALIGN, "depth_metrics: sums and workspace must be 8-byte aligned");
  const size_t need = dusty_depth_metrics_workspace_bytes(p->b, p->h, p->w);
  if (workspace_bytes < need)
    return fail_arg(DUSTY_ENOSPACE, "depth_metrics: workspace %zu < %zu", workspace_bytes, need);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int chunks = chunks_of(p->h, p->w);
  double* partial = static_cast<double*>(workspace);
  depth_chunk_kernel<<<(unsigned)((long long)p->b * chunks), TPB, 0, st>>>(*p, pred, target, out_pred_m, out_target_m,
                                                                           partial, p->h * p->w, chunks);
  DUSTY_AFTER_LAUNCH("depth_chunk_kernel");
  const long long n = (long long)p->b * NSUM;
  depth_combine_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(partial, sums, p->b, chunks);
  DUSTY_AFTER_LAUNCH("depth_combine_kernel");
  return 0;
}
