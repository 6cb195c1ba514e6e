// Fused point-drop head + inverse spherical projection (+ valid-point compaction) for sm_100a.
//
// One streaming pass replaces ~30 element-wise ATen kernels of the reference:
//   GumbelSigmoid.logistic_noise / forward      models/dusty.py:30-59
//   DUSty1.maskout / DUSty2.maskout (eval)      models/dusty.py:77-91, 107-127
//   tanh_to_sigmoid(...).clamp_(0, 1)           utils/__init__.py:76-79, evaluate_synthesis.py:60
//   Coordinate.inv_to_xyz (revert_depth,        utils/lidar.py:23-29, 38-47, 49-56, 61-68
//     normalize/denormalize_minmax, pol_to_xyz)
//   xyz.flatten(2).transpose(1,2) + .contiguous() copies   evaluate_synthesis.py:62, fps/...py:88
//
// Every intermediate is rounded exactly where the reference's separate kernels round it
// (__fadd_rn/__fmul_rn/__fdiv_rn block FMA contraction; expf/logf are the same libdevice
// functions ATen's CUDA kernels call), so masks and points are bit-identical to the reference
// run on the same GPU. HBM traffic per pixel: read depth + confidence, write mask + depth + xyz
// = 28 B (DUSty-I) / 36 B (DUSty-II); the noise map and the trig table are small and L2 resident.
//
// The backward (head_backward_kernel) is the gradient autograd produces through the same chain. It saves nothing:
// it rebuilds every forward value with the forward's helpers from the same inputs and noise, and rounds the chain
// rule where autograd's kernels round it.
#include <algorithm>
#include <cstdlib>

#include "common.cuh"

namespace dusty {
namespace head {

constexpr int TPB = 256;
constexpr int GROUP = TPB * 4;          // pixels per CTA (1024)

// One gate as the kernels read it: its noise (dusty_gate) and its own scalars
struct GateDev {
  int mode;
  int hard;
  const float* a;
  const float* b;
  long long bstride;
  int pstride;
  float inv_tau;
  float eps;
};

struct Args {
  dusty_head_params p;
  GateDev gp, gi;
  const float* depth;
  const float* conf;
  const float* trig;
  float* out_mask;
  float* out_depth;
  float* out_points;
  int* out_count;
  int* out_index;
  float* out_compact;
  unsigned* seg_state;      // one word per CTA: 0x80000000 | count once published
  unsigned* ticket;         // compaction: segments are handed out in the order the CTAs start running
  int npix;                 // h*w
  int segs_per_image;
};

__device__ __forceinline__ float logistic_from_uniform(float u1, float u2, float eps) {
  const float l1 = logf(__fadd_rn(u1, eps));
  const float l2 = logf(__fadd_rn(u2, eps));
  return -logf(__fadd_rn(__fdiv_rn(l1, l2), eps));
}

// GumbelSigmoid.forward of gate g for one logit: the straight-through value, or the soft one when !g.hard.
// The gate is taken by value: a reference into the kernel's parameter costs the 32-register forward kernels 8-16
// more bytes of spills.
__device__ __forceinline__ float gate_value(float logit, const GateDev g, float na, float nb, float threshold) {
  if (g.mode == DUSTY_NOISE_NONE) return logit > 0.0f ? 1.0f : 0.0f;
  const float l = g.mode == DUSTY_NOISE_UNIFORM ? logistic_from_uniform(na, nb, g.eps) : na;
  const float x = __fmul_rn(__fadd_rn(logit, l), g.inv_tau);
  const float soft = __frcp_rn(__fadd_rn(1.0f, expf(-x)));     // == 1.0f / y: both are the correctly rounded quotient
  if (!g.hard) return soft;                                    // GumbelSigmoid(hard=False)
  const float hard = soft > threshold ? 1.0f : 0.0f;           // a NaN threshold gives 0, as in the reference
  return __fadd_rn(__fsub_rn(hard, soft), soft);
}

__device__ __forceinline__ float4 load_noise(const GateDev& g, const float* base, long long img, int pix) {
  // base = g.a or g.b
  const float* q = base + img * g.bstride;
  if (g.pstride == 0) { const float v = q[0]; return make_float4(v, v, v, v); }
  return *reinterpret_cast<const float4*>(q + pix);
}

// inv in [0,1] (NaN passes through) -> normalised range d and validity
__device__ __forceinline__ float range_from_inv(float inv, const dusty_head_params& p, bool& valid) {
  valid = fabsf(inv) > p.tol;
  const float disp = __fadd_rn(__fmul_rn(inv, p.disp_scale), p.disp_shift);
  const float depth = __frcp_rn(disp);                         // == 1.0f / disp, correctly rounded
  const float nrm = __fmul_rn(__fsub_rn(depth, p.min_depth), p.inv_range);
  float d = __fadd_rn(__fmul_rn(nrm, p.range), p.min_depth);
  d = __fmul_rn(d, p.inv_max_depth);
  return __fmul_rn(d, valid ? 1.0f : 0.0f);
}

// One 4-pixel group per thread (32 registers -> 8 CTAs = 2048 threads per SM, 1024 pixels per CTA): occupancy
// hides the latency, the last wave is small (measured against 2 and 4 groups per thread: DESIGN.md 2.1).
//
// Ordered compaction (COMPACT): the valid pixels of an image, in pixel order. A CTA packs its own valid points
// into shared memory (block scan), publishes their number, sums the numbers of the earlier segments of its image
// (one warp reads them in parallel: a single L2 round trip) and copies its packed block to the image's output
// with coalesced stores. The segments of an image are handed out by a per-image ticket counter to the CTAs that
// blockIdx assigns to that image, so every segment a CTA waits for belongs to a CTA that is already running --
// the hardware does not promise to start CTAs in blockIdx order.
template <int C, bool COMPACT>
__global__ void __launch_bounds__(TPB, C == 1 ? 8 : 7) head_project_kernel(const Args a) {
  constexpr int SEG = GROUP;
  // per-warp transpose buffers for the interleaved points (8 x 384 floats); with compaction the same memory then
  // stages the CTA's packed points (3 x 1024 floats) and their pixel indices (1024 ints)
  __shared__ __align__(16) float stage[COMPACT ? 4 * GROUP : (TPB / 32) * 384];
  __shared__ int wsum[TPB / 32];
  __shared__ int s_base;
  const dusty_head_params& p = a.p;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const long long img = blockIdx.x / a.segs_per_image;
  int seg = (int)(blockIdx.x - (unsigned)img * a.segs_per_image);
  if (COMPACT && a.ticket != nullptr) {        // one counter per image, 128 bytes apart: no single hot address
    if (tid == 0) s_base = (int)atomicAdd(a.ticket + img * 32, 1u);
    __syncthreads();
    seg = s_base;
  }
  const int npix = a.npix;

  const float* depth = a.depth + img * npix;
  const float* conf0 = a.conf + img * C * npix;
  float* omask0 = a.out_mask + img * C * npix;
  float* odepth = a.out_depth + img * npix;

  const int pix = seg * SEG + tid * 4;
  unsigned vbits = 0;
  float X[4] = {0.f, 0.f, 0.f, 0.f}, Y[4] = {0.f, 0.f, 0.f, 0.f}, Z[4] = {0.f, 0.f, 0.f, 0.f};
  if (pix < npix) {
    // the streaming loads of this thread first: 2-3 independent 128-bit requests in flight
    const float4 dv = ldg_stream(reinterpret_cast<const float4*>(depth + pix));
    const float4 cv = ldg_stream(reinterpret_cast<const float4*>(conf0 + pix));
    float4 c1 = make_float4(0, 0, 0, 0);
    if (C == 2) c1 = ldg_stream(reinterpret_cast<const float4*>(conf0 + npix + pix));
    float4 na = make_float4(0, 0, 0, 0), nb = na;
    if (a.gp.mode != DUSTY_NOISE_NONE) na = load_noise(a.gp, a.gp.a, img, pix);
    if (a.gp.mode == DUSTY_NOISE_UNIFORM) nb = load_noise(a.gp, a.gp.b, img, pix);
    float mp[4] = {gate_value(cv.x, a.gp, na.x, nb.x, p.threshold), gate_value(cv.y, a.gp, na.y, nb.y, p.threshold),
                   gate_value(cv.z, a.gp, na.z, nb.z, p.threshold), gate_value(cv.w, a.gp, na.w, nb.w, p.threshold)};
    float mk[4] = {mp[0], mp[1], mp[2], mp[3]};
    stg_stream(reinterpret_cast<float4*>(omask0 + pix), make_float4(mp[0], mp[1], mp[2], mp[3]));
    if (C == 2) {
      float4 ia = make_float4(0, 0, 0, 0), ib = ia;
      if (a.gi.mode != DUSTY_NOISE_NONE) ia = load_noise(a.gi, a.gi.a, img, pix);
      if (a.gi.mode == DUSTY_NOISE_UNIFORM) ib = load_noise(a.gi, a.gi.b, img, pix);
      const float mi[4] = {gate_value(c1.x, a.gi, ia.x, ib.x, p.threshold), gate_value(c1.y, a.gi, ia.y, ib.y, p.threshold),
                           gate_value(c1.z, a.gi, ia.z, ib.z, p.threshold), gate_value(c1.w, a.gi, ia.w, ib.w, p.threshold)};
      stg_stream(reinterpret_cast<float4*>(omask0 + npix + pix), make_float4(mi[0], mi[1], mi[2], mi[3]));
      #pragma unroll
      for (int q = 0; q < 4; ++q) mk[q] = __fmul_rn(mp[q], mi[q]);
    }
    const float din[4] = {dv.x, dv.y, dv.z, dv.w};
    float dout[4], rng[4];
    #pragma unroll
    for (int q = 0; q < 4; ++q) {
      // mask * depth + (1 - mask) * drop_const
      dout[q] = __fadd_rn(__fmul_rn(mk[q], din[q]), __fmul_rn(__fsub_rn(1.0f, mk[q]), p.drop_const));
      // tanh_to_sigmoid + clamp_(0,1); NaN survives the clamp as in torch
      float inv = __fmul_rn(__fadd_rn(dout[q], 1.0f), 0.5f);
      inv = inv < 0.0f ? 0.0f : (inv > 1.0f ? 1.0f : inv);
      bool valid;
      rng[q] = range_from_inv(inv, p, valid);
      vbits |= valid ? (1u << q) : 0u;
    }
    stg_stream(reinterpret_cast<float4*>(odepth + pix), make_float4(dout[0], dout[1], dout[2], dout[3]));
    if (COMPACT || a.out_points != nullptr) {                 // maskout alone: no projection, no trig table
      const float4 ce = *reinterpret_cast<const float4*>(a.trig + pix);
      const float4 se = *reinterpret_cast<const float4*>(a.trig + npix + pix);
      const float4 ca = *reinterpret_cast<const float4*>(a.trig + 2 * npix + pix);
      const float4 sa = *reinterpret_cast<const float4*>(a.trig + 3 * npix + pix);
      const float cev[4] = {ce.x, ce.y, ce.z, ce.w}, sev[4] = {se.x, se.y, se.z, se.w};
      const float cav[4] = {ca.x, ca.y, ca.z, ca.w}, sav[4] = {sa.x, sa.y, sa.z, sa.w};
      #pragma unroll
      for (int q = 0; q < 4; ++q) {
        const float rc = __fmul_rn(rng[q], cev[q]);
        X[q] = __fmul_rn(rc, cav[q]);
        Y[q] = __fmul_rn(rc, sav[q]);
        Z[q] = __fmul_rn(rng[q], sev[q]);
      }
      if (a.out_points != nullptr) {
        if (p.points_layout == 0) {
          float* o = a.out_points + img * 3 * npix + pix;
          stg_stream(reinterpret_cast<float4*>(o), make_float4(X[0], X[1], X[2], X[3]));
          stg_stream(reinterpret_cast<float4*>(o + npix), make_float4(Y[0], Y[1], Y[2], Y[3]));
          stg_stream(reinterpret_cast<float4*>(o + 2 * npix), make_float4(Z[0], Z[1], Z[2], Z[3]));
        } else {
          const int wpix = seg * SEG + warp * 128;       // first pixel of this warp's 128
          if (wpix + 128 <= npix) {
            // whole warp in range (uniform): transpose through shared memory so that every STG.128 of
            // the warp covers 512 contiguous bytes instead of 16 bytes out of every 48
            float4* wst = reinterpret_cast<float4*>(stage + warp * 384);
            wst[lane * 3] = make_float4(X[0], Y[0], Z[0], X[1]);
            wst[lane * 3 + 1] = make_float4(Y[1], Z[1], X[2], Y[2]);
            wst[lane * 3 + 2] = make_float4(Z[2], X[3], Y[3], Z[3]);
            __syncwarp();
            float4* o = reinterpret_cast<float4*>(a.out_points + (img * npix + wpix) * 3);
            stg_stream(o + lane, wst[lane]);
            stg_stream(o + lane + 32, wst[lane + 32]);
            stg_stream(o + lane + 64, wst[lane + 64]);
          } else {
            float4* o = reinterpret_cast<float4*>(a.out_points + (img * npix + pix) * 3);
            stg_stream(o, make_float4(X[0], Y[0], Z[0], X[1]));
            stg_stream(o + 1, make_float4(Y[1], Z[1], X[2], Y[2]));
            stg_stream(o + 2, make_float4(Z[2], X[3], Y[3], Z[3]));
          }
        }
      }
    }
  }
  if (!COMPACT) return;

  // ---- ordered compaction ----
  const int c = __popc(vbits);
  int inc = c;
  #pragma unroll
  for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += t; }
  __syncthreads();                       // every warp is done with its transpose buffer (and with s_base)
  if (lane == 31) wsum[warp] = inc;
  __syncthreads();
  int before = 0, cta_total = 0;
  #pragma unroll
  for (int w = 0; w < TPB / 32; ++w) { const int sw = wsum[w]; if (w < warp) before += sw; cta_total += sw; }
  volatile unsigned* st = a.seg_state + img * a.segs_per_image;
  if (tid == 0) st[seg] = 0x80000000u | (unsigned)cta_total;      // the word carries the count itself: nothing to fence
  float* const cxyz = stage;
  int* const cidx = reinterpret_cast<int*>(stage + 3 * GROUP);
  int pos = before + inc - c;
  #pragma unroll
  for (int q = 0; q < 4; ++q) {
    if (vbits & (1u << q)) {
      cxyz[3 * pos] = X[q]; cxyz[3 * pos + 1] = Y[q]; cxyz[3 * pos + 2] = Z[q];
      cidx[pos] = pix + q;
      ++pos;
    }
  }
  if (warp == 0) {                       // earlier segments of this image, 32 at a time, in parallel
    int base = 0;
    for (int s0 = 0; s0 < seg; s0 += 32) {
      unsigned v = 0x80000000u;
      if (s0 + lane < seg) {               // back off between polls: a spinning warp must not take issue slots and LSU
        v = st[s0 + lane];                 // bandwidth from the CTAs it is waiting for
        while (!(v & 0x80000000u)) { __nanosleep(64); v = st[s0 + lane]; }
      }
      base += (int)__reduce_add_sync(0xffffffffu, v & 0x7fffffffu);
    }
    if (lane == 0) {
      s_base = base;
      if (seg == a.segs_per_image - 1 && a.out_count) a.out_count[img] = base + cta_total;
    }
  }
  __syncthreads();
  const long long first = img * npix + s_base;
  if (a.out_compact) {
    float* o = a.out_compact + first * 3;
    for (int i = tid; i < 3 * cta_total; i += TPB) o[i] = cxyz[i];
  }
  if (a.out_index) {
    int* o = a.out_index + first;
    for (int i = tid; i < cta_total; i += TPB) o[i] = cidx[i];
  }
}

// Compaction for large batches: one CTA of 512 threads owns a whole image and walks it in 2048-pixel steps with the
// next step's loads already in flight, so the running number of valid pixels never leaves the CTA: no look-back,
// no tickets, no waiting on other CTAs (the segment kernel above spends its time exactly there: each CTA is a
// chain of ticket -> loads -> count -> look-back -> copy, and only a few CTAs fit an SM). Every warp packs its
// valid points through its own shared-memory buffer and writes them with coalesced stores. Used when the batch
// alone fills the GPU (b >= 128 images); the arithmetic is the same code as above, bit for bit.
constexpr int IMG_TPB = 512;
constexpr int IMG_STEP = IMG_TPB * 4;                    // pixels per step
constexpr int IMG_TABLE_BYTES = 2 * 5 * IMG_STEP * 4;    // two stages of {cos el, sin el, cos az, sin az, noise} tiles (80 KB)

template <int C>
__global__ void __launch_bounds__(IMG_TPB, 2) head_project_image_kernel(const Args a) {
  constexpr int NWARP = IMG_TPB / 32;
  __shared__ __align__(16) float stage[NWARP * 384];      // per-warp: transpose of 128 points, then its packed points
  __shared__ int istage[NWARP * 128];                     // per-warp: pixel indices of its packed points
  __shared__ int wsum[2][NWARP];
  __shared__ uint64_t full[2];
  // The trig table and the (per-pixel, logistic) noise map are L2 resident and shared by all images; loading them
  // where they are used puts two dependent L2 round trips into every step of a CTA that has only 16 warps. They
  // are therefore brought in one step ahead by 1-D TMA bulk copies (no registers held across the step).
  extern __shared__ __align__(128) float tables[];
  const dusty_head_params& p = a.p;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const long long img = blockIdx.x;
  const int npix = a.npix;
  const bool noise_tile = a.gp.mode == DUSTY_NOISE_LOGISTIC && a.gp.pstride == 1;
  auto prefetch_tables = [&](int step) {                 // one thread; stage = step & 1
    float* dst = tables + (step & 1) * (5 * IMG_STEP);
    const int first = step * IMG_STEP;
    const uint32_t bytes = (uint32_t)min(IMG_STEP, npix - first) * 4u;
    mbar_expect_tx(&full[step & 1], (noise_tile ? 5u : 4u) * bytes);
    #pragma unroll
    for (int t = 0; t < 4; ++t) bulk_g2s(dst + t * IMG_STEP, a.trig + (long long)t * npix + first, bytes, &full[step & 1]);
    if (noise_tile) bulk_g2s(dst + 4 * IMG_STEP, a.gp.a + img * a.gp.bstride + first, bytes, &full[step & 1]);
  };
  if (tid == 0) { mbar_init(&full[0], 1); mbar_init(&full[1], 1); mbar_fence_init(); }
  __syncthreads();
  if (tid == 0) prefetch_tables(0);
  const float* depth = a.depth + img * npix;
  const float* conf0 = a.conf + img * C * npix;
  float* omask0 = a.out_mask + img * C * npix;
  float* odepth = a.out_depth + img * npix;
  float* const wst = stage + warp * 384;
  int* const wix = istage + warp * 128;
  const int steps = (npix + IMG_TPB * 4 - 1) / (IMG_TPB * 4);

  float4 dv = make_float4(0, 0, 0, 0), cv = dv, c1 = dv;
  if (tid * 4 < npix) {
    dv = ldg_stream(reinterpret_cast<const float4*>(depth + tid * 4));
    cv = ldg_stream(reinterpret_cast<const float4*>(conf0 + tid * 4));
    if (C == 2) c1 = ldg_stream(reinterpret_cast<const float4*>(conf0 + npix + tid * 4));
  }
  int running = 0;
  for (int it = 0; it < steps; ++it) {
    const int pix = it * (IMG_TPB * 4) + tid * 4;
    const float4 dcur = dv, ccur = cv, c1cur = c1;
    // every thread is past the previous step's barrier, hence done with the stage that is refilled now
    if (tid == 0 && it + 1 < steps) prefetch_tables(it + 1);
    mbar_wait(&full[it & 1], (uint32_t)((it >> 1) & 1));
    const float* const tab = tables + (it & 1) * (5 * IMG_STEP) + tid * 4;
    const int nxt = pix + IMG_TPB * 4;
    if (it + 1 < steps && nxt < npix) {                   // next step's streaming loads
      dv = ldg_stream(reinterpret_cast<const float4*>(depth + nxt));
      cv = ldg_stream(reinterpret_cast<const float4*>(conf0 + nxt));
      if (C == 2) c1 = ldg_stream(reinterpret_cast<const float4*>(conf0 + npix + nxt));
    }
    unsigned vbits = 0;
    float X[4] = {0.f, 0.f, 0.f, 0.f}, Y[4] = {0.f, 0.f, 0.f, 0.f}, Z[4] = {0.f, 0.f, 0.f, 0.f};
    if (pix < npix) {
      float4 na = make_float4(0, 0, 0, 0), nb = na;
      if (noise_tile) na = *reinterpret_cast<const float4*>(tab + 4 * IMG_STEP);
      else if (a.gp.mode != DUSTY_NOISE_NONE) na = load_noise(a.gp, a.gp.a, img, pix);
      if (a.gp.mode == DUSTY_NOISE_UNIFORM) nb = load_noise(a.gp, a.gp.b, img, pix);
      float mp[4] = {gate_value(ccur.x, a.gp, na.x, nb.x, p.threshold), gate_value(ccur.y, a.gp, na.y, nb.y, p.threshold),
                     gate_value(ccur.z, a.gp, na.z, nb.z, p.threshold), gate_value(ccur.w, a.gp, na.w, nb.w, p.threshold)};
      float mk[4] = {mp[0], mp[1], mp[2], mp[3]};
      stg_stream(reinterpret_cast<float4*>(omask0 + pix), make_float4(mp[0], mp[1], mp[2], mp[3]));
      if (C == 2) {
        float4 ia = make_float4(0, 0, 0, 0), ib = ia;
        if (a.gi.mode != DUSTY_NOISE_NONE) ia = load_noise(a.gi, a.gi.a, img, pix);
        if (a.gi.mode == DUSTY_NOISE_UNIFORM) ib = load_noise(a.gi, a.gi.b, img, pix);
        const float mi[4] = {gate_value(c1cur.x, a.gi, ia.x, ib.x, p.threshold), gate_value(c1cur.y, a.gi, ia.y, ib.y, p.threshold),
                             gate_value(c1cur.z, a.gi, ia.z, ib.z, p.threshold), gate_value(c1cur.w, a.gi, ia.w, ib.w, p.threshold)};
        stg_stream(reinterpret_cast<float4*>(omask0 + npix + pix), make_float4(mi[0], mi[1], mi[2], mi[3]));
        #pragma unroll
        for (int q = 0; q < 4; ++q) mk[q] = __fmul_rn(mp[q], mi[q]);
      }
      const float din[4] = {dcur.x, dcur.y, dcur.z, dcur.w};
      float dout[4], rng[4];
      #pragma unroll
      for (int q = 0; q < 4; ++q) {
        dout[q] = __fadd_rn(__fmul_rn(mk[q], din[q]), __fmul_rn(__fsub_rn(1.0f, mk[q]), p.drop_const));
        float inv = __fmul_rn(__fadd_rn(dout[q], 1.0f), 0.5f);
        inv = inv < 0.0f ? 0.0f : (inv > 1.0f ? 1.0f : inv);
        bool valid;
        rng[q] = range_from_inv(inv, p, valid);
        vbits |= valid ? (1u << q) : 0u;
      }
      stg_stream(reinterpret_cast<float4*>(odepth + pix), make_float4(dout[0], dout[1], dout[2], dout[3]));
      const float4 ce = *reinterpret_cast<const float4*>(tab);
      const float4 se = *reinterpret_cast<const float4*>(tab + IMG_STEP);
      const float4 ca = *reinterpret_cast<const float4*>(tab + 2 * IMG_STEP);
      const float4 sa = *reinterpret_cast<const float4*>(tab + 3 * IMG_STEP);
      const float cev[4] = {ce.x, ce.y, ce.z, ce.w}, sev[4] = {se.x, se.y, se.z, se.w};
      const float cav[4] = {ca.x, ca.y, ca.z, ca.w}, sav[4] = {sa.x, sa.y, sa.z, sa.w};
      #pragma unroll
      for (int q = 0; q < 4; ++q) {
        const float rc = __fmul_rn(rng[q], cev[q]);
        X[q] = __fmul_rn(rc, cav[q]);
        Y[q] = __fmul_rn(rc, sav[q]);
        Z[q] = __fmul_rn(rng[q], sev[q]);
      }
    }
    const int wpix = it * (IMG_TPB * 4) + warp * 128;     // first pixel of this warp's 128
    if (a.out_points != nullptr) {
      if (p.points_layout == 0) {
        if (pix < npix) {
          float* o = a.out_points + img * 3 * npix + pix;
          stg_stream(reinterpret_cast<float4*>(o), make_float4(X[0], X[1], X[2], X[3]));
          stg_stream(reinterpret_cast<float4*>(o + npix), make_float4(Y[0], Y[1], Y[2], Y[3]));
          stg_stream(reinterpret_cast<float4*>(o + 2 * npix), make_float4(Z[0], Z[1], Z[2], Z[3]));
        }
      } else if (wpix + 128 <= npix) {                    // warp-uniform
        float4* w4 = reinterpret_cast<float4*>(wst);
        w4[lane * 3] = make_float4(X[0], Y[0], Z[0], X[1]);
        w4[lane * 3 + 1] = make_float4(Y[1], Z[1], X[2], Y[2]);
        w4[lane * 3 + 2] = make_float4(Z[2], X[3], Y[3], Z[3]);
        __syncwarp();
        float4* o = reinterpret_cast<float4*>(a.out_points + (img * npix + wpix) * 3);
        stg_stream(o + lane, w4[lane]);
        stg_stream(o + lane + 32, w4[lane + 32]);
        stg_stream(o + lane + 64, w4[lane + 64]);
        __syncwarp();
      } else if (pix < npix) {
        float4* o = reinterpret_cast<float4*>(a.out_points + (img * npix + pix) * 3);
        stg_stream(o, make_float4(X[0], Y[0], Z[0], X[1]));
        stg_stream(o + 1, make_float4(Y[1], Z[1], X[2], Y[2]));
        stg_stream(o + 2, make_float4(Z[2], X[3], Y[3], Z[3]));
      }
    }
    // ---- ordered compaction: warp scan, one barrier per step (double-buffered warp sums), packed warp stores ----
    const int c = __popc(vbits);
    int inc = c;
    #pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += t; }
    const int wcount = __shfl_sync(0xffffffffu, inc, 31);
    if (lane == 31) wsum[it & 1][warp] = inc;
    int off = inc - c;
    #pragma unroll
    for (int q = 0; q < 4; ++q) {
      if (vbits & (1u << q)) {
        wst[3 * off] = X[q]; wst[3 * off + 1] = Y[q]; wst[3 * off + 2] = Z[q];
        wix[off] = pix + q;
        ++off;
      }
    }
    __syncthreads();
    int ws = lane < NWARP ? wsum[it & 1][lane] : 0;       // inclusive scan of the 16 warp sums by shuffles
    #pragma unroll
    for (int o = 1; o < NWARP; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, ws, o); if (lane >= o) ws += t; }
    const int total = __shfl_sync(0xffffffffu, ws, NWARP - 1);
    const int before = warp == 0 ? 0 : __shfl_sync(0xffffffffu, ws, warp - 1);
    const long long first = img * npix + running + before;
    if (a.out_compact) {
      float* o = a.out_compact + first * 3;
      for (int i = lane; i < 3 * wcount; i += 32) o[i] = wst[i];
    }
    if (a.out_index) {
      int* o = a.out_index + first;
      for (int i = lane; i < wcount; i += 32) o[i] = wix[i];
    }
    __syncwarp();
    running += total;
  }
  if (tid == 0 && a.out_count) a.out_count[img] = running;
}

__global__ void __launch_bounds__(TPB) inv_to_xyz_kernel(const dusty_head_params p, const float* __restrict__ inv_all,
                                                         const float* __restrict__ trig, float* __restrict__ out, int npix) {
  const long long img = blockIdx.y;
  const int pix = (blockIdx.x * TPB + threadIdx.x) * 4;
  if (pix >= npix) return;
  const float4 iv = ldg_stream(reinterpret_cast<const float4*>(inv_all + img * npix + pix));
  const float in[4] = {iv.x, iv.y, iv.z, iv.w};
  const float4 ce = *reinterpret_cast<const float4*>(trig + pix);
  const float4 se = *reinterpret_cast<const float4*>(trig + npix + pix);
  const float4 ca = *reinterpret_cast<const float4*>(trig + 2 * npix + pix);
  const float4 sa = *reinterpret_cast<const float4*>(trig + 3 * npix + pix);
  const float cev[4] = {ce.x, ce.y, ce.z, ce.w}, sev[4] = {se.x, se.y, se.z, se.w};
  const float cav[4] = {ca.x, ca.y, ca.z, ca.w}, sav[4] = {sa.x, sa.y, sa.z, sa.w};
  float X[4], Y[4], Z[4];
  #pragma unroll
  for (int q = 0; q < 4; ++q) {
    bool valid;
    const float r = range_from_inv(in[q], p, valid);
    const float rc = __fmul_rn(r, cev[q]);
    X[q] = __fmul_rn(rc, cav[q]);
    Y[q] = __fmul_rn(rc, sav[q]);
    Z[q] = __fmul_rn(r, sev[q]);
  }
  if (p.points_layout == 0) {
    float* o = out + img * 3 * npix + pix;
    stg_stream(reinterpret_cast<float4*>(o), make_float4(X[0], X[1], X[2], X[3]));
    stg_stream(reinterpret_cast<float4*>(o + npix), make_float4(Y[0], Y[1], Y[2], Y[3]));
    stg_stream(reinterpret_cast<float4*>(o + 2 * npix), make_float4(Z[0], Z[1], Z[2], Z[3]));
  } else {
    float4* o = reinterpret_cast<float4*>(out + (img * npix + pix) * 3);
    stg_stream(o, make_float4(X[0], Y[0], Z[0], X[1]));
    stg_stream(o + 1, make_float4(Y[1], Z[1], X[2], Y[2]));
    stg_stream(o + 2, make_float4(Z[2], X[3], Y[3], Z[3]));
  }
}

__global__ void __launch_bounds__(TPB) logistic_noise_kernel(const float* __restrict__ u1, const float* __restrict__ u2,
                                                             float eps, size_t count, float* __restrict__ out) {
  for (size_t i = (size_t)blockIdx.x * TPB + threadIdx.x; i < count; i += (size_t)gridDim.x * TPB)
    out[i] = logistic_from_uniform(u1[i], u2[i], eps);
}

__global__ void __launch_bounds__(TPB) gumbel_sigmoid_kernel(const float* __restrict__ logits, const GateDev g,
                                                             float threshold, int npix, float* __restrict__ out) {
  const long long img = blockIdx.y;
  const int pix = (blockIdx.x * TPB + threadIdx.x) * 4;
  if (pix >= npix) return;
  const float4 cv = ldg_stream(reinterpret_cast<const float4*>(logits + img * npix + pix));
  float4 na = make_float4(0, 0, 0, 0), nb = na;
  if (g.mode != DUSTY_NOISE_NONE) na = load_noise(g, g.a, img, pix);
  if (g.mode == DUSTY_NOISE_UNIFORM) nb = load_noise(g, g.b, img, pix);
  stg_stream(reinterpret_cast<float4*>(out + img * npix + pix),
             make_float4(gate_value(cv.x, g, na.x, nb.x, threshold), gate_value(cv.y, g, na.y, nb.y, threshold),
                         gate_value(cv.z, g, na.z, nb.z, threshold), gate_value(cv.w, g, na.w, nb.w, threshold)));
}

// ---- backward of head_project_kernel ----
struct BwdArgs {
  dusty_head_params p;
  GateDev gp, gi;
  const float* depth;
  const float* conf;
  const float* trig;
  const float* grad_mask;     // (b,C,h,w) or NULL
  const float* grad_depth;    // (b,1,h,w) or NULL
  const float* grad_points;   // layout p.points_layout; NULL unless the PROJ instantiation runs
  float* grad_depth_in;
  float* grad_conf;
  float* tau_partial;         // per gate, one float per CTA (pixel gate, then image gate), or NULL when d/d inv_tau is not wanted
  int npix;
  int segs_per_image;
};

// Gradient of gate gt's GumbelSigmoid with respect to its logit, given the gradient g of its (straight-through or
// soft) output. The soft value is rebuilt from the same noise and in the same rounding as gate_value. The term
// d soft / d inv_tau is added to the gate's own accumulator tau; a gate without noise is (logit > 0): no gradient.
__device__ __forceinline__ float gate_grad(float logit, const GateDev gt, float na, float nb, float g, float& tau) {
  if (gt.mode == DUSTY_NOISE_NONE) return 0.0f;
  const float l = gt.mode == DUSTY_NOISE_UNIFORM ? logistic_from_uniform(na, nb, gt.eps) : na;
  const float xl = __fadd_rn(logit, l);
  const float soft = __frcp_rn(__fadd_rn(1.0f, expf(-__fmul_rn(xl, gt.inv_tau))));
  const float gx = __fmul_rn(__fmul_rn(g, __fsub_rn(1.0f, soft)), soft);     // ATen sigmoid_backward: (g * (1 - y)) * y
  tau = __fadd_rn(tau, __fmul_rn(gx, xl));
  return __fmul_rn(gx, gt.inv_tau);
}

__device__ __forceinline__ float4 ldg_or_zero(const float* base, long long off) {
  return base ? ldg_stream(reinterpret_cast<const float4*>(base + off)) : make_float4(0, 0, 0, 0);
}

// One 4-pixel group per thread, the forward's grid. Every forward value (gates, mask, dout, inv, validity) is
// recomputed with the forward's helpers from the same inputs and noise, hence bit-identical to what the forward
// returned. PROJ adds the projection's gradient; interleaved grad_points arrive through the forward's per-warp
// transpose run backwards (coalesced 512-byte loads per warp instruction).
template <int C, bool PROJ>
__global__ void __launch_bounds__(TPB, PROJ ? 3 : 4) head_backward_kernel(const BwdArgs a) {
  __shared__ __align__(16) float stage[PROJ ? (TPB / 32) * 384 : 4];
  __shared__ float wtau[C][TPB / 32];
  const dusty_head_params& p = a.p;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const long long img = blockIdx.x / a.segs_per_image;
  const int seg = (int)(blockIdx.x - (unsigned)img * a.segs_per_image);
  const int npix = a.npix;
  const int pix = seg * GROUP + tid * 4;
  float tau_p = 0.0f, tau_i = 0.0f;         // d/d inv_tau of the pixel and the image gate
  float4 gpx = make_float4(0, 0, 0, 0), gpy = gpx, gpz = gpx;
  if (PROJ) {
    if (p.points_layout == 0) {
      if (pix < npix) {
        const float* g = a.grad_points + img * 3 * npix + pix;
        gpx = ldg_stream(reinterpret_cast<const float4*>(g));
        gpy = ldg_stream(reinterpret_cast<const float4*>(g + npix));
        gpz = ldg_stream(reinterpret_cast<const float4*>(g + 2 * npix));
      }
    } else {
      const int wpix = seg * GROUP + warp * 128;
      float4 v0 = make_float4(0, 0, 0, 0), v1 = v0, v2 = v0;
      if (wpix + 128 <= npix) {                         // whole warp in range (uniform)
        const float4* g = reinterpret_cast<const float4*>(a.grad_points + (img * npix + wpix) * 3);
        float4* wst = reinterpret_cast<float4*>(stage + warp * 384);
        wst[lane] = ldg_stream(g + lane);
        wst[lane + 32] = ldg_stream(g + lane + 32);
        wst[lane + 64] = ldg_stream(g + lane + 64);
        __syncwarp();
        v0 = wst[lane * 3]; v1 = wst[lane * 3 + 1]; v2 = wst[lane * 3 + 2];
      } else if (pix < npix) {
        const float4* g = reinterpret_cast<const float4*>(a.grad_points + (img * npix + pix) * 3);
        v0 = ldg_stream(g); v1 = ldg_stream(g + 1); v2 = ldg_stream(g + 2);
      }
      gpx = make_float4(v0.x, v0.w, v1.z, v2.y);
      gpy = make_float4(v0.y, v1.x, v1.w, v2.z);
      gpz = make_float4(v0.z, v1.y, v2.x, v2.w);
    }
  }
  if (pix < npix) {
    const float* conf0 = a.conf + img * C * npix;
    const float4 dv = ldg_stream(reinterpret_cast<const float4*>(a.depth + img * npix + pix));
    const float4 cv = ldg_stream(reinterpret_cast<const float4*>(conf0 + pix));
    const float4 c1 = C == 2 ? ldg_stream(reinterpret_cast<const float4*>(conf0 + npix + pix)) : make_float4(0, 0, 0, 0);
    const float4 gd = ldg_or_zero(a.grad_depth, img * npix + pix);
    const float4 gm0 = ldg_or_zero(a.grad_mask, img * C * npix + pix);
    const float4 gm1 = C == 2 ? ldg_or_zero(a.grad_mask, img * C * npix + npix + pix) : make_float4(0, 0, 0, 0);
    float4 na = make_float4(0, 0, 0, 0), nb = na, ia = na, ib = na;
    if (a.gp.mode != DUSTY_NOISE_NONE) na = load_noise(a.gp, a.gp.a, img, pix);
    if (a.gp.mode == DUSTY_NOISE_UNIFORM) nb = load_noise(a.gp, a.gp.b, img, pix);
    if (C == 2 && a.gi.mode != DUSTY_NOISE_NONE) ia = load_noise(a.gi, a.gi.a, img, pix);
    if (C == 2 && a.gi.mode == DUSTY_NOISE_UNIFORM) ib = load_noise(a.gi, a.gi.b, img, pix);
    const float din[4] = {dv.x, dv.y, dv.z, dv.w}, cp[4] = {cv.x, cv.y, cv.z, cv.w}, ci[4] = {c1.x, c1.y, c1.z, c1.w};
    const float gdv[4] = {gd.x, gd.y, gd.z, gd.w}, gmp[4] = {gm0.x, gm0.y, gm0.z, gm0.w}, gmi[4] = {gm1.x, gm1.y, gm1.z, gm1.w};
    const float nav[4] = {na.x, na.y, na.z, na.w}, nbv[4] = {nb.x, nb.y, nb.z, nb.w};
    const float iav[4] = {ia.x, ia.y, ia.z, ia.w}, ibv[4] = {ib.x, ib.y, ib.z, ib.w};
    float grng[4] = {0.f, 0.f, 0.f, 0.f};
    if (PROJ) {
      // d/d range of ((r cos el) cos az, (r cos el) sin az, r sin el): autograd's operand order, and the order in
      // which its engine adds the three branches (z, then y, then x)
      const float4 ce = *reinterpret_cast<const float4*>(a.trig + pix);
      const float4 se = *reinterpret_cast<const float4*>(a.trig + npix + pix);
      const float4 ca = *reinterpret_cast<const float4*>(a.trig + 2 * npix + pix);
      const float4 sa = *reinterpret_cast<const float4*>(a.trig + 3 * npix + pix);
      const float cev[4] = {ce.x, ce.y, ce.z, ce.w}, sev[4] = {se.x, se.y, se.z, se.w};
      const float cav[4] = {ca.x, ca.y, ca.z, ca.w}, sav[4] = {sa.x, sa.y, sa.z, sa.w};
      const float gx[4] = {gpx.x, gpx.y, gpx.z, gpx.w}, gy[4] = {gpy.x, gpy.y, gpy.z, gpy.w}, gz[4] = {gpz.x, gpz.y, gpz.z, gpz.w};
      #pragma unroll
      for (int q = 0; q < 4; ++q)
        grng[q] = __fadd_rn(__fadd_rn(__fmul_rn(gz[q], sev[q]), __fmul_rn(__fmul_rn(gy[q], sav[q]), cev[q])),
                            __fmul_rn(__fmul_rn(gx[q], cav[q]), cev[q]));
    }
    float gdin[4], gc0[4], gc1[4];
    #pragma unroll
    for (int q = 0; q < 4; ++q) {
      const float mp = gate_value(cp[q], a.gp, nav[q], nbv[q], p.threshold);
      const float mi = C == 2 ? gate_value(ci[q], a.gi, iav[q], ibv[q], p.threshold) : 1.0f;
      const float mk = C == 2 ? __fmul_rn(mp, mi) : mp;
      float gdout = gdv[q];
      if (PROJ) {
        const float dout = __fadd_rn(__fmul_rn(mk, din[q]), __fmul_rn(__fsub_rn(1.0f, mk), p.drop_const));
        const float pre = __fmul_rn(__fadd_rn(dout, 1.0f), 0.5f);
        const float inv = pre < 0.0f ? 0.0f : (pre > 1.0f ? 1.0f : pre);
        bool valid;
        range_from_inv(inv, p, valid);
        const float rcp = __frcp_rn(__fadd_rn(__fmul_rn(inv, p.disp_scale), p.disp_shift));
        float g = __fmul_rn(grng[q], valid ? 1.0f : 0.0f);
        g = __fmul_rn(__fmul_rn(__fmul_rn(g, p.inv_max_depth), p.range), p.inv_range);
        g = __fmul_rn(-g, __fmul_rn(rcp, rcp));                       // reciprocal_backward: -g * (y * y)
        g = __fmul_rn(g, p.disp_scale);
        g = (pre >= 0.0f && pre <= 1.0f) ? g : 0.0f;                  // clamp_backward keeps the bounds
        gdout = __fadd_rn(gdout, __fmul_rn(g, 0.5f));
      }
      gdin[q] = __fmul_rn(gdout, mk);
      // d/d mask of mask * depth + (1 - mask) * drop_const; DUSty-I adds it to the mask's own gradient in the order
      // autograd does: (grad_mask - g * drop_const) + g * depth
      const float gdrop = __fmul_rn(gdout, p.drop_const), gblend = __fmul_rn(gdout, din[q]);
      if (C == 1) {
        gc0[q] = gate_grad(cp[q], a.gp, nav[q], nbv[q], __fadd_rn(__fsub_rn(gmp[q], gdrop), gblend), tau_p);
      } else {
        const float gm = __fsub_rn(gblend, gdrop);
        gc0[q] = gate_grad(cp[q], a.gp, nav[q], nbv[q], __fadd_rn(__fmul_rn(gm, mi), gmp[q]), tau_p);
        gc1[q] = gate_grad(ci[q], a.gi, iav[q], ibv[q], __fadd_rn(__fmul_rn(gm, mp), gmi[q]), tau_i);
      }
    }
    float* gco = a.grad_conf + img * C * npix + pix;
    stg_stream(reinterpret_cast<float4*>(a.grad_depth_in + img * npix + pix), make_float4(gdin[0], gdin[1], gdin[2], gdin[3]));
    stg_stream(reinterpret_cast<float4*>(gco), make_float4(gc0[0], gc0[1], gc0[2], gc0[3]));
    if (C == 2) stg_stream(reinterpret_cast<float4*>(gco + npix), make_float4(gc1[0], gc1[1], gc1[2], gc1[3]));
  }
  if (a.tau_partial == nullptr) return;
  // per-CTA partial of d/d inv_tau for each gate: fixed shuffle tree, then the 8 warp sums in warp order
  #pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    tau_p = __fadd_rn(tau_p, __shfl_xor_sync(0xffffffffu, tau_p, o));
    if (C == 2) tau_i = __fadd_rn(tau_i, __shfl_xor_sync(0xffffffffu, tau_i, o));
  }
  if (lane == 0) {
    wtau[0][warp] = tau_p;
    if (C == 2) wtau[C - 1][warp] = tau_i;
  }
  __syncthreads();
  if (tid < C) {                         // thread 0: pixel gate, thread 1: image gate
    float s = 0.0f;
    #pragma unroll
    for (int w = 0; w < TPB / 32; ++w) s = __fadd_rn(s, wtau[tid][w]);
    a.tau_partial[tid * gridDim.x + blockIdx.x] = s;
  }
}

// d/d inv_tau of gate blockIdx.x = sum of its n per-CTA partials: one CTA per gate, fixed order (strided per thread,
// then a fixed tree), in double.
__global__ void __launch_bounds__(TPB) head_backward_tau_kernel(const float* __restrict__ partial, int n, float* __restrict__ out) {
  __shared__ double s[TPB];
  partial += (long long)blockIdx.x * n;
  double acc = 0.0;
  for (int i = threadIdx.x; i < n; i += TPB) acc += (double)partial[i];
  s[threadIdx.x] = acc;
  __syncthreads();
  for (int o = TPB / 2; o > 0; o >>= 1) {
    if (threadIdx.x < o) s[threadIdx.x] += s[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) out[blockIdx.x] = (float)s[0];
}

static int check_params(const dusty_head_params* p, const char* who) {
  if (!p) return fail_arg(DUSTY_EINVAL, "%s: null params", who);
  if (p->b < 0 || p->h <= 0 || p->w <= 0) return fail_arg(DUSTY_EINVAL, "%s: bad shape b=%d h=%d w=%d", who, p->b, p->h, p->w);
  if (p->w % 4 != 0) return fail_arg(DUSTY_EINVAL, "%s: w=%d must be a multiple of 4", who, p->w);
  if ((long long)p->h * p->w > 0x7fffffffLL / 4) return fail_arg(DUSTY_EINVAL, "%s: image too large", who);
  if (p->points_layout != 0 && p->points_layout != 1) return fail_arg(DUSTY_EINVAL, "%s: points_layout must be 0 or 1", who);
  return 0;
}

static int check_gate(const dusty_gate& g, const char* name) {
  if (g.mode < DUSTY_NOISE_NONE || g.mode > DUSTY_NOISE_UNIFORM) return fail_arg(DUSTY_EINVAL, "head_project: %s gate mode %d", name, g.mode);
  if (g.hard != 0 && g.hard != 1) return fail_arg(DUSTY_EINVAL, "head_project: %s gate hard must be 0 or 1", name);
  if (g.mode != DUSTY_NOISE_NONE && !g.noise_a) return fail_arg(DUSTY_EINVAL, "head_project: %s gate needs noise_a", name);
  if (g.mode == DUSTY_NOISE_UNIFORM && !g.noise_b) return fail_arg(DUSTY_EINVAL, "head_project: %s gate needs noise_b", name);
  if (g.pixel_stride != 0 && g.pixel_stride != 1) return fail_arg(DUSTY_EINVAL, "head_project: %s gate pixel_stride must be 0 or 1", name);
  if (g.mode != DUSTY_NOISE_NONE && g.pixel_stride == 1) {
    if (!aligned16(g.noise_a) || (g.noise_b && !aligned16(g.noise_b)) || (g.batch_stride % 4) != 0)
      return fail_arg(DUSTY_EALIGN, "head_project: %s gate noise must be 16-byte aligned with batch_stride %% 4 == 0", name);
  }
  return 0;
}

static GateDev gate_dev(const dusty_gate& g) {
  return GateDev{g.mode, g.hard, g.noise_a, g.noise_b, g.batch_stride, (int)g.pixel_stride, g.inv_tau, g.eps};
}

}  // namespace head
}  // namespace dusty

using namespace dusty;
using namespace dusty::head;

extern "C" size_t dusty_head_project_workspace_bytes(int b, int h, int w) {
  if (b <= 0 || h <= 0 || w <= 0) return 0;
  const long long npix = (long long)h * w;
  const long long segs = (npix + GROUP - 1) / GROUP;      // the finest segmentation any launch uses
  return align_up(((size_t)b * segs + (size_t)b * 32) * sizeof(unsigned), 256);      // segment states + per-image ticket counters
}

extern "C" int dusty_head_project(const dusty_head_params* p, const float* depth, const float* confidence,
                                  const float* trig, float* out_mask, float* out_depth, float* out_points,
                                  int32_t* out_count, int32_t* out_index, float* out_compact, void* workspace,
                                  size_t workspace_bytes, void* stream) {
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (int rc = check_params(p, "head_project")) return rc;
  if (p->conf_channels != 1 && p->conf_channels != 2) return fail_arg(DUSTY_EINVAL, "head_project: conf_channels must be 1 or 2");
  if (p->b == 0) return 0;
  if (int rc = check_device()) return rc;
  const bool compact = out_count || out_index || out_compact;
  if (!depth || !confidence || !out_mask || !out_depth || (!trig && (out_points || compact)))
    return fail_arg(DUSTY_EINVAL, "head_project: null pointer");
  if (!aligned16(depth) || !aligned16(confidence) || (trig && !aligned16(trig)) || !aligned16(out_mask) || !aligned16(out_depth) ||
      (out_points && !aligned16(out_points)))
    return fail_arg(DUSTY_EALIGN, "head_project: tensors must be 16-byte aligned");
  if (int rc = check_gate(p->gate_pixel, "pixel")) return rc;
  if (p->conf_channels == 2) if (int rc = check_gate(p->gate_image, "image")) return rc;
  Args a{};
  a.p = *p;
  a.gp = gate_dev(p->gate_pixel);
  a.gi = gate_dev(p->gate_image);
  if (p->conf_channels == 1) a.gi.mode = DUSTY_NOISE_NONE;
  a.depth = depth; a.conf = confidence; a.trig = trig;
  a.out_mask = out_mask; a.out_depth = out_depth; a.out_points = out_points;
  a.out_count = out_count; a.out_index = out_index; a.out_compact = out_compact;
  a.npix = p->h * p->w;
  a.segs_per_image = (a.npix + GROUP - 1) / GROUP;
  const long long ctas = (long long)p->b * a.segs_per_image;
  if (ctas > 0x7fffffffLL) return fail_arg(DUSTY_EINVAL, "head_project: grid too large");
  // batches that fill the GPU with one CTA per image: no cross-CTA scan at all (DUSTY_HEAD_COMPACT=segment|image forces one)
  const char* const forced = getenv("DUSTY_HEAD_COMPACT");
  const int force_path = !forced ? 0 : (forced[0] == 's' ? 1 : (forced[0] == 'i' ? 2 : 0));
  if (compact && (force_path == 2 || (force_path == 0 && p->b >= 128))) {
    static bool configured[kMaxDevices] = {};
    const int dev = current_device();
    if (!configured[dev]) {
      DUSTY_CUDA(cudaFuncSetAttribute(head_project_image_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, IMG_TABLE_BYTES));
      DUSTY_CUDA(cudaFuncSetAttribute(head_project_image_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, IMG_TABLE_BYTES));
      configured[dev] = true;
    }
    if (p->conf_channels == 1) head_project_image_kernel<1><<<(unsigned)p->b, IMG_TPB, IMG_TABLE_BYTES, st>>>(a);
    else head_project_image_kernel<2><<<(unsigned)p->b, IMG_TPB, IMG_TABLE_BYTES, st>>>(a);
    DUSTY_AFTER_LAUNCH("head_project_image_kernel");
    return 0;
  }
  if (compact) {
    if (!workspace || workspace_bytes < dusty_head_project_workspace_bytes(p->b, p->h, p->w))
      return fail_arg(DUSTY_ENOSPACE, "head_project: compaction needs %zu workspace bytes", dusty_head_project_workspace_bytes(p->b, p->h, p->w));
    a.seg_state = static_cast<unsigned*>(workspace);
    a.ticket = a.seg_state + ctas;
    static const bool no_ticket = [] { const char* e = getenv("DUSTY_HEAD_TICKET"); return e && e[0] == '0'; }();   // A/B only
    DUSTY_CUDA(cudaMemsetAsync(workspace, 0, ((size_t)ctas + (size_t)p->b * 32) * sizeof(unsigned), st));
    if (no_ticket) a.ticket = nullptr;
  }
  if (p->conf_channels == 1) {
    if (compact) head_project_kernel<1, true><<<(unsigned)ctas, TPB, 0, st>>>(a);
    else head_project_kernel<1, false><<<(unsigned)ctas, TPB, 0, st>>>(a);
  } else {
    if (compact) head_project_kernel<2, true><<<(unsigned)ctas, TPB, 0, st>>>(a);
    else head_project_kernel<2, false><<<(unsigned)ctas, TPB, 0, st>>>(a);
  }
  DUSTY_AFTER_LAUNCH("head_project_kernel");
  return 0;
}

extern "C" size_t dusty_head_project_backward_workspace_bytes(int b, int h, int w) {
  if (b <= 0 || h <= 0 || w <= 0) return 0;
  const long long segs = ((long long)h * w + GROUP - 1) / GROUP;
  return align_up(2 * (size_t)b * segs * sizeof(float), 256);      // one partial of d/d inv_tau per gate and CTA
}

extern "C" int dusty_head_project_backward(const dusty_head_params* p, const float* depth, const float* confidence,
                                           const float* trig, const float* grad_mask, const float* grad_depth,
                                           const float* grad_points, float* grad_depth_in, float* grad_confidence,
                                           float* grad_inv_tau, void* workspace, size_t workspace_bytes, void* stream) {
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (int rc = check_params(p, "head_project_backward")) return rc;
  if (p->conf_channels != 1 && p->conf_channels != 2)
    return fail_arg(DUSTY_EINVAL, "head_project_backward: conf_channels must be 1 or 2");
  if (p->b == 0) return 0;
  if (!depth || !confidence || !grad_depth_in || !grad_confidence || (grad_points && !trig))
    return fail_arg(DUSTY_EINVAL, "head_project_backward: null pointer");
  if (!aligned16(depth) || !aligned16(confidence) || (trig && !aligned16(trig)) || !aligned16(grad_mask) ||
      !aligned16(grad_depth) || !aligned16(grad_points) || !aligned16(grad_depth_in) || !aligned16(grad_confidence))
    return fail_arg(DUSTY_EALIGN, "head_project_backward: tensors must be 16-byte aligned");
  if (int rc = check_gate(p->gate_pixel, "pixel")) return rc;
  if (p->conf_channels == 2) if (int rc = check_gate(p->gate_image, "image")) return rc;
  const size_t ws_need = dusty_head_project_backward_workspace_bytes(p->b, p->h, p->w);
  if (grad_inv_tau && (!workspace || workspace_bytes < ws_need))
    return fail_arg(DUSTY_ENOSPACE, "head_project_backward: grad_inv_tau needs %zu workspace bytes", ws_need);
  BwdArgs a{};
  a.p = *p;
  a.gp = gate_dev(p->gate_pixel);
  a.gi = gate_dev(p->gate_image);
  if (p->conf_channels == 1) a.gi.mode = DUSTY_NOISE_NONE;
  a.depth = depth; a.conf = confidence; a.trig = trig;
  a.grad_mask = grad_mask; a.grad_depth = grad_depth; a.grad_points = grad_points;
  a.grad_depth_in = grad_depth_in; a.grad_conf = grad_confidence;
  a.tau_partial = grad_inv_tau ? static_cast<float*>(workspace) : nullptr;
  a.npix = p->h * p->w;
  a.segs_per_image = (a.npix + GROUP - 1) / GROUP;
  const long long ctas = (long long)p->b * a.segs_per_image;
  if (ctas > 0x7fffffffLL) return fail_arg(DUSTY_EINVAL, "head_project_backward: grid too large");
  if (int rc = check_device()) return rc;
  const bool proj = grad_points != nullptr;
  if (p->conf_channels == 1) {
    if (proj) head_backward_kernel<1, true><<<(unsigned)ctas, TPB, 0, st>>>(a);
    else head_backward_kernel<1, false><<<(unsigned)ctas, TPB, 0, st>>>(a);
  } else {
    if (proj) head_backward_kernel<2, true><<<(unsigned)ctas, TPB, 0, st>>>(a);
    else head_backward_kernel<2, false><<<(unsigned)ctas, TPB, 0, st>>>(a);
  }
  DUSTY_AFTER_LAUNCH("head_backward_kernel");
  if (grad_inv_tau) {
    head_backward_tau_kernel<<<(unsigned)p->conf_channels, TPB, 0, st>>>(a.tau_partial, (int)ctas, grad_inv_tau);
    DUSTY_AFTER_LAUNCH("head_backward_tau_kernel");
  }
  return 0;
}

extern "C" int dusty_gumbel_sigmoid(const float* logits, const dusty_gate* gate, float threshold, int b, int npix, float* out,
                                    void* stream) {
  if (b < 0 || npix <= 0 || npix % 4 != 0) return fail_arg(DUSTY_EINVAL, "gumbel_sigmoid: bad shape b=%d npix=%d", b, npix);
  if (b == 0) return 0;
  if (b > 65535) return fail_arg(DUSTY_EINVAL, "gumbel_sigmoid: batch %d exceeds 65535", b);
  if (int rc = check_device()) return rc;
  if (!logits || !gate || !out) return fail_arg(DUSTY_EINVAL, "gumbel_sigmoid: null pointer");
  if (!aligned16(logits) || !aligned16(out)) return fail_arg(DUSTY_EALIGN, "gumbel_sigmoid: tensors must be 16-byte aligned");
  if (int rc = check_gate(*gate, "gumbel")) return rc;
  gumbel_sigmoid_kernel<<<dim3((npix / 4 + TPB - 1) / TPB, b), TPB, 0, static_cast<cudaStream_t>(stream)>>>(
      logits, gate_dev(*gate), threshold, npix, out);
  DUSTY_AFTER_LAUNCH("gumbel_sigmoid_kernel");
  return 0;
}

extern "C" int dusty_inv_to_xyz(const dusty_head_params* p, const float* inv, const float* trig, float* out_points,
                                void* stream) {
  if (int rc = check_params(p, "inv_to_xyz")) return rc;
  if (p->b == 0) return 0;
  if (p->b > 65535) return fail_arg(DUSTY_EINVAL, "inv_to_xyz: batch %d exceeds 65535", p->b);
  if (int rc = check_device()) return rc;
  if (!inv || !trig || !out_points) return fail_arg(DUSTY_EINVAL, "inv_to_xyz: null pointer");
  if (!aligned16(inv) || !aligned16(trig) || !aligned16(out_points)) return fail_arg(DUSTY_EALIGN, "inv_to_xyz: tensors must be 16-byte aligned");
  const int npix = p->h * p->w;
  inv_to_xyz_kernel<<<dim3((npix / 4 + TPB - 1) / TPB, p->b), TPB, 0, static_cast<cudaStream_t>(stream)>>>(*p, inv, trig, out_points, npix);
  DUSTY_AFTER_LAUNCH("inv_to_xyz_kernel");
  return 0;
}

extern "C" int dusty_logistic_noise(const float* u1, const float* u2, float eps, size_t count, float* out, void* stream) {
  if (count == 0) return 0;
  if (int rc = check_device()) return rc;
  if (!u1 || !u2 || !out) return fail_arg(DUSTY_EINVAL, "logistic_noise: null pointer");
  const unsigned grid = (unsigned)std::min<size_t>((count + TPB - 1) / TPB, (size_t)kNumSMs * 16);
  logistic_noise_kernel<<<grid, TPB, 0, static_cast<cudaStream_t>(stream)>>>(u1, u2, eps, count, out);
  DUSTY_AFTER_LAUNCH("logistic_noise_kernel");
  return 0;
}
