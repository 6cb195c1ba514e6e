// Sliced Wasserstein distance between two sets of range images (SURVEY.md §3a: compute_swd of the reference's
// evaluate_synthesis.py) for sm_100a. The algorithm is Karras et al.'s SWD as the swd-pytorch port publishes it
// (DESIGN.md §2.7 states the contract step by step).
//
// Stage A (dusty_swd_descriptors), per image set:
//   swd_down_kernel   G(l+1) = conv2d(G(l), binomial 5x5 / 256, padding 2, stride 2) per plane, into the workspace;
//   swd_patch_kernel  one CTA per (image, level): the Laplacian G(l) - conv2d(up2(G(l+1)), k, padding 2) is evaluated
//                     only at the 7x7 patches of the sampled positions and written once as descriptor rows; the CTA
//                     also reduces its (mean, M2) per channel in double;
//   swd_stats_kernel  combines the per-image (mean, M2) in a fixed order (Chan et al.) -> (mean, unbiased std).
// Stage B (dusty_swd_sliced), per level, for batches of directions:
//   swd_project_kernel  normalises a tile of rows on load ((x - mean) / (std + 1e-8), f32) and projects it onto 32
//                       directions with one fixed FMA order, writing order-preserving u32 keys;
//   swd_radix_kernel    one CTA sorts one (set, direction) segment: an LSD radix sort of four 8-bit passes, stable
//                       ranks from warp ballots (linear in the segment length whatever the key distribution);
//   swd_absdiff_kernel  one CTA per direction: sum_i |a_(i) - b_(i)| in double in a fixed order.
// Nothing is reduced with atomics on floating-point values, so two calls give bit-identical sums, and each direction's
// sum does not depend on which other directions share its batch or its rank.
#include "common.cuh"

#include <vector>

namespace dusty {
namespace swd {

constexpr int kPatch = 7;
constexpr int kPatch2 = kPatch * kPatch;
constexpr int kMaxLevels = 16;
constexpr int kMaxChannels = 4;
constexpr int TPB = 256;
constexpr int kProjRows = 128;          // rows per projection CTA (one per thread)
constexpr int kProjDirs = 32;           // directions per projection CTA (register accumulators)
constexpr int kSortThreads = 512;
constexpr int kSortWarps = kSortThreads / 32;
constexpr long long kMaxRows = 1LL << 30;
constexpr size_t kKeyBudget = size_t(4) << 30;   // bytes of keys (both sets, both sort buffers) per direction batch

// The binomial [1,4,6,4,1] / 16 per axis: the 5x5 kernel of the reference is the outer product (exact in f32).
__device__ __forceinline__ float binom(int i) { return i == 2 ? 0.375f : (i == 1 || i == 3) ? 0.25f : 0.0625f; }

struct Levels {
  const float* g[kMaxLevels];   // G(l), (n, c, h_l, w_l)
  float* desc[kMaxLevels];      // (n * n_desc, c * 49)
  int h[kMaxLevels], w[kMaxLevels];
};

__global__ void __launch_bounds__(TPB) swd_down_kernel(const float* __restrict__ src, float* __restrict__ dst,
                                                       long long planes, int h, int w) {
  const int ho = h >> 1, wo = w >> 1;
  const long long total = planes * ho * wo;
  for (long long e = blockIdx.x * (long long)TPB + threadIdx.x; e < total; e += (long long)gridDim.x * TPB) {
    const long long plane = e / ((long long)ho * wo);
    const int rem = (int)(e - plane * ho * wo), y = rem / wo, x = rem - y * wo;
    const float* s = src + plane * h * w;
    float acc = 0.f;
    #pragma unroll
    for (int i = 0; i < 5; ++i) {
      const int sy = 2 * y + i - 2;
      if (sy < 0 || sy >= h) continue;
      #pragma unroll
      for (int j = 0; j < 5; ++j) {
        const int sx = 2 * x + j - 2;
        if (sx < 0 || sx >= w) continue;
        acc = fmaf(binom(i) * binom(j), s[(long long)sy * w + sx], acc);
      }
    }
    dst[e] = acc;
  }
}

// Laplacian level l of one plane at (y, x): G(l)(y,x) - sum k(i,j) up2(G(l+1))(y+i-2, x+j-2), zero padded.
__device__ __forceinline__ float laplacian(const float* __restrict__ g, const float* __restrict__ gn, int h, int w,
                                           int y, int x, bool last) {
  const float v = g[(long long)y * w + x];
  if (last) return v;
  const int wn = w >> 1;
  float acc = 0.f;
  #pragma unroll
  for (int i = 0; i < 5; ++i) {
    const int uy = y + i - 2;
    if (uy < 0 || uy >= h) continue;
    #pragma unroll
    for (int j = 0; j < 5; ++j) {
      const int ux = x + j - 2;
      if (ux < 0 || ux >= w) continue;
      acc = fmaf(binom(i) * binom(j), gn[(long long)(uy >> 1) * wn + (ux >> 1)], acc);
    }
  }
  return v - acc;
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

// grid (n, levels): descriptors of image blockIdx.x at level blockIdx.y, and their (mean, M2) per channel into
// partial[((level * c + ch) * n + image) * 2 + {0, 1}].
__global__ void __launch_bounds__(TPB) swd_patch_kernel(Levels lv, int levels, int n, int c,
                                                        const int* __restrict__ positions, int n_desc,
                                                        double* __restrict__ partial) {
  __shared__ double sm[TPB / 32];
  const int img = blockIdx.x, l = blockIdx.y;
  const int h = lv.h[l], w = lv.w[l], span = w - (kPatch - 1), K = c * kPatch2;
  const bool last = l == levels - 1;
  const int* pos = positions + (long long)l * n_desc;
  float* out = lv.desc[l] + (long long)img * n_desc * K;
  const int count = n_desc * kPatch2;
  for (int ch = 0; ch < c; ++ch) {
    const float* g = lv.g[l] + ((long long)img * c + ch) * h * w;
    const float* gn = last ? nullptr : lv.g[l + 1] + ((long long)img * c + ch) * (h >> 1) * (w >> 1);
    double s = 0.0;
    for (int t = threadIdx.x; t < count; t += TPB) {
      const int d = t / kPatch2, r = t - d * kPatch2, p = pos[d];
      const int py = p / span, px = p - py * span;
      const float v = laplacian(g, gn, h, w, py + r / kPatch, px + r % kPatch, last);
      out[(long long)d * K + ch * kPatch2 + r] = v;
      s += (double)v;
    }
    const double mean = block_sum(s, sm) / (double)count;
    double m2 = 0.0;
    for (int t = threadIdx.x; t < count; t += TPB) {     // each thread re-reads what it wrote above
      const int d = t / kPatch2, r = t - d * kPatch2;
      const double e = (double)out[(long long)d * K + ch * kPatch2 + r] - mean;
      m2 += e * e;
    }
    m2 = block_sum(m2, sm);
    if (threadIdx.x == 0) {
      double* dst = partial + (((long long)l * c + ch) * n + img) * 2;
      dst[0] = mean;
      dst[1] = m2;
    }
    __syncthreads();
  }
}

// Chan et al.'s pairwise update of (count, mean, M2). A constant set keeps mean exact and M2 = 0.
__device__ __forceinline__ void chan(double& cnt, double& mean, double& m2, double cb, double mb, double m2b) {
  if (cb == 0.0) return;
  if (cnt == 0.0) { cnt = cb; mean = mb; m2 = m2b; return; }
  const double tot = cnt + cb, delta = mb - mean;
  mean += delta * (cb / tot);
  m2 += m2b + delta * delta * (cnt * cb / tot);
  cnt = tot;
}

// grid (levels * c): stats[(l * c + ch) * 2 + {0, 1}] = mean, unbiased std over all images.
__global__ void __launch_bounds__(TPB) swd_stats_kernel(const double* __restrict__ partial, int n, double per_image,
                                                        double* __restrict__ stats) {
  __shared__ double s_cnt[TPB], s_mean[TPB], s_m2[TPB];
  const double* p = partial + (long long)blockIdx.x * n * 2;
  const int chunk = (n + TPB - 1) / TPB, lo = threadIdx.x * chunk, hi = min(n, lo + chunk);
  double cnt = 0.0, mean = 0.0, m2 = 0.0;
  for (int i = lo; i < hi; ++i) chan(cnt, mean, m2, per_image, p[2 * i], p[2 * i + 1]);
  s_cnt[threadIdx.x] = cnt; s_mean[threadIdx.x] = mean; s_m2[threadIdx.x] = m2;
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int t = 1; t < TPB; ++t) chan(cnt, mean, m2, s_cnt[t], s_mean[t], s_m2[t]);
    stats[2 * blockIdx.x] = mean;
    stats[2 * blockIdx.x + 1] = sqrt(m2 / (cnt - 1.0));
  }
}

// Order-preserving f32 <-> u32 (ascending float order is ascending key order; -0 sorts just below +0).
__device__ __forceinline__ uint32_t f2key(float f) {
  const uint32_t b = __float_as_uint(f);
  return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
__device__ __forceinline__ float key2f(uint32_t k) {
  return __uint_as_float((k & 0x80000000u) ? (k ^ 0x80000000u) : ~k);
}

struct ProjectArgs {
  const float* desc[2];
  const double* stats[2];      // (c, 2): mean, std
  const float* dirs;           // (K, n_dirs)
  int n_dirs, dir_first, dir_stride, batch;   // direction of batch slot j: dir_first + j * dir_stride
  int rows, c;
  uint32_t* keys;              // (2, batch, rows)
};

// grid (ceil(rows / 128), ceil(batch / 32), 2 sets), 128 threads; dynamic smem (K * 32 + K * 129) floats.
__global__ void __launch_bounds__(kProjRows) swd_project_kernel(ProjectArgs a) {
  extern __shared__ float smem[];
  const int K = a.c * kPatch2, set = blockIdx.z;
  float* s_w = smem;                         // [K][kProjDirs], 16-byte rows
  float* s_x = smem + K * kProjDirs;         // [K][kProjRows + 1]
  __shared__ float s_mean[kMaxChannels], s_den[kMaxChannels];
  __shared__ int s_nan[kProjRows];          // a row with a NaN component projects to NaN on every direction
  s_nan[threadIdx.x] = 0;
  const double* stats = set ? a.stats[1] : a.stats[0];      // (a.stats[set] would copy the parameters to the stack)
  if (threadIdx.x < a.c) {
    s_mean[threadIdx.x] = (float)stats[2 * threadIdx.x];
    s_den[threadIdx.x] = __fadd_rn((float)stats[2 * threadIdx.x + 1], 1e-8f);
  }
  const int row0 = blockIdx.x * kProjRows, j0 = blockIdx.y * kProjDirs;
  const int nrows = min(kProjRows, a.rows - row0), ndirs = min(kProjDirs, a.batch - j0);
  for (int e = threadIdx.x; e < K * kProjDirs; e += kProjRows) {
    const int k = e / kProjDirs, j = e - k * kProjDirs;
    s_w[e] = j < ndirs ? a.dirs[(long long)k * a.n_dirs + a.dir_first + (long long)(j0 + j) * a.dir_stride] : 0.f;
  }
  __syncthreads();
  const float* src = (set ? a.desc[1] : a.desc[0]) + (long long)row0 * K;
  for (int e = threadIdx.x; e < kProjRows * K; e += kProjRows) {
    const int r = e / K, k = e - r * K, ch = k / kPatch2;
    float v = 0.f;
    if (r < nrows) v = __fdiv_rn(__fsub_rn(src[e], s_mean[ch]), s_den[ch]);
    if (isnan(v)) s_nan[r] = 1;
    s_x[k * (kProjRows + 1) + r] = v;
  }
  __syncthreads();
  float acc[kProjDirs];
  #pragma unroll
  for (int j = 0; j < kProjDirs; ++j) acc[j] = -0.f;   // -0 + p = p for every p: a row of -0 products projects to -0
  for (int k = 0; k < K; ++k) {
    const float x = s_x[k * (kProjRows + 1) + threadIdx.x];
    const float4* w4 = reinterpret_cast<const float4*>(s_w + k * kProjDirs);
    #pragma unroll
    for (int q = 0; q < kProjDirs / 4; ++q) {
      const float4 w = w4[q];
      acc[4 * q + 0] = fmaf(w.x, x, acc[4 * q + 0]);
      acc[4 * q + 1] = fmaf(w.y, x, acc[4 * q + 1]);
      acc[4 * q + 2] = fmaf(w.z, x, acc[4 * q + 2]);
      acc[4 * q + 3] = fmaf(w.w, x, acc[4 * q + 3]);
    }
  }
  if (threadIdx.x < nrows) {
    const bool nan_row = s_nan[threadIdx.x] != 0;
    uint32_t* dst = a.keys + ((long long)set * a.batch + j0) * a.rows + row0 + threadIdx.x;
    #pragma unroll
    for (int j = 0; j < kProjDirs; ++j)
      if (j < ndirs) dst[(long long)j * a.rows] = nan_row ? 0xffffffffu : f2key(acc[j]);
  }
}

// Lanes of this warp whose 9-bit digit equals mine (bit 8 marks lanes past the segment's end).
__device__ __forceinline__ uint32_t peers_of(uint32_t digit) {
  uint32_t peers = 0xffffffffu;
  #pragma unroll
  for (int b = 0; b < 9; ++b) {
    const uint32_t bal = __ballot_sync(0xffffffffu, (digit >> b) & 1u);
    peers &= ((digit >> b) & 1u) ? bal : ~bal;
  }
  return peers;
}

// grid (2 * batch): segment blockIdx.x of keys (rows each) is sorted ascending in place; alt is scratch of the
// same size. Four stable 8-bit passes: keys -> alt -> keys -> alt -> keys.
__global__ void __launch_bounds__(kSortThreads) swd_radix_kernel(uint32_t* __restrict__ keys, uint32_t* __restrict__ alt,
                                                                 int rows) {
  __shared__ uint32_t s_hist[4][256];
  __shared__ uint32_t s_cnt[kSortWarps][256];
  __shared__ uint32_t s_off[kSortWarps][256];
  __shared__ uint32_t s_base[256];
  const long long seg = (long long)blockIdx.x * rows;
  uint32_t* bufs[2] = {keys + seg, alt + seg};
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const uint32_t lt = (1u << lane) - 1u;
  for (int e = threadIdx.x; e < 4 * 256; e += kSortThreads) (&s_hist[0][0])[e] = 0u;
  for (int e = threadIdx.x; e < kSortWarps * 256; e += kSortThreads) (&s_cnt[0][0])[e] = 0u;
  __syncthreads();
  // the four digit histograms in one read
  for (int base = 0; base < rows; base += kSortThreads) {
    const int i = base + threadIdx.x;
    const bool valid = i < rows;
    const uint32_t key = valid ? bufs[0][i] : 0u;
    #pragma unroll
    for (int p = 0; p < 4; ++p) {
      const uint32_t digit = valid ? (key >> (8 * p)) & 255u : 256u;
      const uint32_t peers = peers_of(digit);
      if (valid && (peers & lt) == 0u) atomicAdd(&s_hist[p][digit], (uint32_t)__popc(peers));
    }
  }
  __syncthreads();
  if (threadIdx.x < 4) {
    uint32_t run = 0;
    for (int d = 0; d < 256; ++d) { const uint32_t c = s_hist[threadIdx.x][d]; s_hist[threadIdx.x][d] = run; run += c; }
  }
  __syncthreads();
  for (int p = 0; p < 4; ++p) {
    const uint32_t* src = bufs[p & 1];
    uint32_t* dst = bufs[(p + 1) & 1];
    if (threadIdx.x < 256) s_base[threadIdx.x] = s_hist[p][threadIdx.x];
    for (int base = 0; base < rows; base += kSortThreads) {
      const int i = base + threadIdx.x;
      const bool valid = i < rows;
      const uint32_t key = valid ? src[i] : 0u;
      const uint32_t digit = valid ? (key >> (8 * p)) & 255u : 256u;
      const uint32_t peers = peers_of(digit);
      if (valid && (peers & lt) == 0u) s_cnt[warp][digit] = __popc(peers);
      __syncthreads();
      if (threadIdx.x < 256) {
        uint32_t run = s_base[threadIdx.x];
        #pragma unroll
        for (int w = 0; w < kSortWarps; ++w) {
          const uint32_t c = s_cnt[w][threadIdx.x];
          s_cnt[w][threadIdx.x] = 0u;
          s_off[w][threadIdx.x] = run;
          run += c;
        }
        s_base[threadIdx.x] = run;
      }
      __syncthreads();
      if (valid) dst[s_off[warp][digit] + __popc(peers & lt)] = key;
    }
    __syncthreads();
  }
}

// grid (batch): sums[dir_first + j * dir_stride] = sum_i |a_(i) - b_(i)| of direction slot j, in double.
__global__ void __launch_bounds__(TPB) swd_absdiff_kernel(const uint32_t* __restrict__ keys, int rows, int batch,
                                                          int dir_first, int dir_stride, double* __restrict__ sums) {
  __shared__ double sm[TPB / 32];
  const uint32_t* a = keys + (long long)blockIdx.x * rows;
  const uint32_t* b = keys + ((long long)batch + blockIdx.x) * rows;
  double s = 0.0;
  for (int i = threadIdx.x; i < rows; i += TPB) s += fabs((double)key2f(a[i]) - (double)key2f(b[i]));
  s = block_sum(s, sm);
  if (threadIdx.x == 0) sums[dir_first + (long long)blockIdx.x * dir_stride] = s;
}

// ---- host side ----

size_t pyramid_floats(int n, int c, int h, int w, int levels) {
  size_t f = 0;
  for (int l = 1; l < levels; ++l) f += (size_t)n * c * (size_t)(h >> l) * (size_t)(w >> l);
  return f;
}

int check_shape(const char* who, int n, int c, int h, int w, int levels, int n_desc) {
  if (n <= 0 || h <= 0 || w <= 0) return fail_arg(DUSTY_EINVAL, "%s: bad sizes n=%d h=%d w=%d", who, n, h, w);
  if (c < 1 || c > kMaxChannels) return fail_arg(DUSTY_EINVAL, "%s: c=%d channels (1..4 supported)", who, c);
  if (levels < 1 || levels > kMaxLevels) return fail_arg(DUSTY_EINVAL, "%s: levels=%d (1..%d)", who, levels, kMaxLevels);
  if (n_desc < 1) return fail_arg(DUSTY_EINVAL, "%s: n_desc=%d must be positive", who, n_desc);
  if ((long long)h * w > 0x7fffffffLL || (long long)n * c > 0x7fffffffLL || (long long)n * n_desc > kMaxRows ||
      (long long)n_desc * c * kPatch2 > 0x7fffffffLL)
    return fail_arg(DUSTY_EINVAL, "%s: sizes n=%d c=%d h=%d w=%d n_desc=%d overflow the kernels' indexing", who, n, c, h,
                    w, n_desc);
  const int f = 1 << (levels - 1);
  if (h % f || w % f)
    return fail_arg(DUSTY_EINVAL, "%s: %dx%d is not divisible by 2^(levels-1) = %d", who, h, w, f);
  for (int l = 0; l < levels; ++l) {
    const int hl = h >> l, wl = w >> l;
    if (hl < kPatch || wl < kPatch)
      return fail_arg(DUSTY_EINVAL, "%s: level %d is %dx%d, smaller than the 7x7 patch", who, l, hl, wl);
    if ((long long)(hl - 6) * (wl - 6) < n_desc)
      return fail_arg(DUSTY_EINVAL, "%s: level %d (%dx%d) has %lld patch positions, fewer than n_desc=%d", who, l, hl,
                      wl, (long long)(hl - 6) * (wl - 6), n_desc);
  }
  return 0;
}

int check_sliced(int rows, int c, int n_dirs, int dir_begin, int dir_end, int dir_stride) {
  if (rows < 1 || rows > kMaxRows) return fail_arg(DUSTY_EINVAL, "swd_sliced: rows=%d (1..2^30)", rows);
  if (c < 1 || c > kMaxChannels) return fail_arg(DUSTY_EINVAL, "swd_sliced: c=%d channels (1..4 supported)", c);
  if (n_dirs < 1) return fail_arg(DUSTY_EINVAL, "swd_sliced: n_dirs=%d must be positive", n_dirs);
  if (dir_begin < 0 || dir_end > n_dirs || dir_stride < 1)
    return fail_arg(DUSTY_EINVAL, "swd_sliced: bad direction range [%d,%d) stride %d of %d", dir_begin, dir_end,
                    dir_stride, n_dirs);
  return 0;
}

// Directions per batch: as many as kKeyBudget allows, balanced over the batches that `count` directions need.
int batch_of(int rows, int count) {
  long long cap = (long long)(kKeyBudget / (16ull * (size_t)rows));
  if (cap < 1) cap = 1;
  const long long nbat = (count + cap - 1) / cap;
  return (int)((count + nbat - 1) / nbat);
}

int set_smem(const void* fn, size_t bytes) {
  static size_t configured[kMaxDevices] = {};
  const int dev = current_device();
  if (bytes > configured[dev]) {
    DUSTY_CUDA(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
    configured[dev] = bytes;
  }
  return 0;
}

}  // namespace swd
}  // namespace dusty

using namespace dusty;
using namespace dusty::swd;

extern "C" size_t dusty_swd_descriptors_workspace_bytes(int n, int c, int h, int w, int levels, int n_desc) {
  if (n <= 0 || c <= 0 || h <= 0 || w <= 0 || levels <= 0 || levels > kMaxLevels || n_desc <= 0) return 0;
  return align_up(sizeof(float) * pyramid_floats(n, c, h, w, levels), 256) + sizeof(double) * 2 * (size_t)levels * c * n;
}

extern "C" int dusty_swd_descriptors(const float* images, int n, int c, int h, int w, int levels,
                                     const int32_t* positions, int n_desc, float* desc, double* stats, void* ws,
                                     size_t ws_bytes, void* stream) {
  if (int rc = check_shape("swd_descriptors", n, c, h, w, levels, n_desc)) return rc;
  if (int rc = check_device()) return rc;
  if (!images || !positions || !desc || !stats || !ws) return fail_arg(DUSTY_EINVAL, "swd_descriptors: null pointer");
  const size_t need = dusty_swd_descriptors_workspace_bytes(n, c, h, w, levels, n_desc);
  if (ws_bytes < need) return fail_arg(DUSTY_ENOSPACE, "swd_descriptors: workspace %zu < %zu", ws_bytes, need);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  // The positions index the patches: checked on the host before any kernel reads through them.
  std::vector<int32_t> host((size_t)levels * n_desc);
  DUSTY_CUDA(cudaMemcpyAsync(host.data(), positions, sizeof(int32_t) * host.size(), cudaMemcpyDefault, st));
  DUSTY_CUDA(cudaStreamSynchronize(st));
  for (int l = 0; l < levels; ++l) {
    const long long np = (long long)((h >> l) - 6) * ((w >> l) - 6);
    for (int d = 0; d < n_desc; ++d) {
      const int32_t p = host[(size_t)l * n_desc + d];
      if (p < 0 || p >= np)
        return fail_arg(DUSTY_EINVAL, "swd_descriptors: position %d of level %d is %d, outside [0, %lld)", d, l, p, np);
    }
  }
  Levels lv{};
  float* pyr = static_cast<float*>(ws);
  const long long planes = (long long)n * c;
  const size_t K = (size_t)c * kPatch2;
  for (int l = 0; l < levels; ++l) {
    lv.h[l] = h >> l;
    lv.w[l] = w >> l;
    lv.desc[l] = desc + (size_t)l * n * n_desc * K;
    if (l == 0) {
      lv.g[0] = images;
    } else {
      lv.g[l] = pyr;
      const long long out = planes * lv.h[l] * lv.w[l];
      const long long blocks = (out + TPB - 1) / TPB;
      swd_down_kernel<<<(int)(blocks < 65535LL * 16 ? blocks : 65535LL * 16), TPB, 0, st>>>(lv.g[l - 1], pyr, planes,
                                                                                          lv.h[l - 1], lv.w[l - 1]);
      DUSTY_AFTER_LAUNCH("swd_down_kernel");
      pyr += out;
    }
  }
  double* partial = reinterpret_cast<double*>(static_cast<char*>(ws) +
                                              align_up(sizeof(float) * pyramid_floats(n, c, h, w, levels), 256));
  swd_patch_kernel<<<dim3(n, levels), TPB, 0, st>>>(lv, levels, n, c, positions, n_desc, partial);
  DUSTY_AFTER_LAUNCH("swd_patch_kernel");
  swd_stats_kernel<<<levels * c, TPB, 0, st>>>(partial, n, (double)n_desc * kPatch2, stats);
  DUSTY_AFTER_LAUNCH("swd_stats_kernel");
  return 0;
}

extern "C" size_t dusty_swd_sliced_workspace_bytes(int rows, int c, int n_dirs) {
  if (rows <= 0 || rows > kMaxRows || c <= 0 || n_dirs <= 0) return 0;
  return 16ull * (size_t)rows * (size_t)batch_of(rows, n_dirs);
}

extern "C" int dusty_swd_sliced(const float* desc1, const float* desc2, const double* stats1, const double* stats2,
                                int rows, int c, const float* dirs, int n_dirs, int dir_begin, int dir_end,
                                int dir_stride, double* sums, void* ws, size_t ws_bytes, void* stream) {
  if (int rc = check_sliced(rows, c, n_dirs, dir_begin, dir_end, dir_stride)) return rc;
  if (dir_begin >= dir_end) return 0;
  if (int rc = check_device()) return rc;
  if (!desc1 || !desc2 || !stats1 || !stats2 || !dirs || !sums || !ws)
    return fail_arg(DUSTY_EINVAL, "swd_sliced: null pointer");
  const size_t need = dusty_swd_sliced_workspace_bytes(rows, c, n_dirs);
  if (ws_bytes < need) return fail_arg(DUSTY_ENOSPACE, "swd_sliced: workspace %zu < %zu", ws_bytes, need);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int K = c * kPatch2;
  const size_t smem = sizeof(float) * (size_t)K * (kProjRows + 1 + kProjDirs);
  if (int rc = set_smem(reinterpret_cast<const void*>(swd_project_kernel), smem)) return rc;
  const int owned = (dir_end - dir_begin + dir_stride - 1) / dir_stride;
  // batch_of is not monotone in its count: a call owning fewer directions than n_dirs may balance to a larger batch
  // than the workspace query sized, so the batch is capped at the queried one.
  const int sized = batch_of(rows, n_dirs), balanced = batch_of(rows, owned);
  const int per = balanced < sized ? balanced : sized;
  uint32_t* keys = static_cast<uint32_t*>(ws);
  uint32_t* alt = keys + 2ull * (size_t)per * rows;
  for (int j0 = 0; j0 < owned; j0 += per) {
    const int cnt = owned - j0 < per ? owned - j0 : per;
    ProjectArgs a{};
    a.desc[0] = desc1; a.desc[1] = desc2; a.stats[0] = stats1; a.stats[1] = stats2;
    a.dirs = dirs; a.n_dirs = n_dirs; a.dir_first = dir_begin + j0 * dir_stride; a.dir_stride = dir_stride;
    a.batch = cnt; a.rows = rows; a.c = c; a.keys = keys;
    const dim3 grid((rows + kProjRows - 1) / kProjRows, (cnt + kProjDirs - 1) / kProjDirs, 2);
    swd_project_kernel<<<grid, kProjRows, smem, st>>>(a);
    DUSTY_AFTER_LAUNCH("swd_project_kernel");
    swd_radix_kernel<<<2 * cnt, kSortThreads, 0, st>>>(keys, alt, rows);
    DUSTY_AFTER_LAUNCH("swd_radix_kernel");
    swd_absdiff_kernel<<<cnt, TPB, 0, st>>>(keys, rows, cnt, a.dir_first, dir_stride, sums);
    DUSTY_AFTER_LAUNCH("swd_absdiff_kernel");
  }
  return 0;
}
