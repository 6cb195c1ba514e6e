// Resident-pair Chamfer search for the evaluation's own shape (clouds of at most PAIR_CAP points, k-d ordered by
// prep_sort_kernel<true>): included by chamfer.cu inside namespace dusty::chamfer.
//
// One CTA per matrix entry keeps BOTH clouds (scan format, 32 KB each at 2048 points) and their chunk boxes in shared
// memory -- one round of four TMA bulk copies per entry instead of a tile stream per row block -- and its warps take
// (direction, row group) tasks from a shared counter. A row group is 32 consecutive rows of the k-d order, i.e. one
// leaf of the row cloud's tree. For its group a warp
//   1. bounds every candidate chunk from below by the distance between the chunk's box and the leaf's box (two
//      chunks per lane) and keeps the bounds as sortable keys;
//   2. visits chunks BEST FIRST (one REDUX.MIN per pick): the nearest chunks tighten every row's running minimum
//      immediately, and the walk ends at the first chunk whose bound exceeds the largest running minimum of the group;
//   3. scans a picked chunk only if some row's own distance to the chunk's box is within that row's running minimum;
//   4. finishes like nn_kernel's DEFERRED pass: the winning 8-candidate window of every row is re-evaluated in the
//      reference's rounding, and a runner-up window inside the search's error window sends the row through an exact
//      scan of every chunk its box bound cannot exclude.
// Every bound is the reference's own distance formula on per-axis gaps (monotone, so it never exceeds a rounded pair
// distance: oracle property test tests/test_oracle_golden.py), hence the results are the brute-force kernel's bit for
// bit.
//
// The scan is bound by FFMA2/FMNMX3 dispatch (8.9 cycles per row and candidate pair), so the way to go faster is to
// evaluate fewer pairs: on the bench's 2048-point FPS clouds 32-row groups visit 8.3 % of the pairs against 11.0 % for
// 64-row groups. With one row per lane, though, every candidate pair costs two warp-uniform LDS.128 = four
// shared-memory wavefronts per four arithmetic instructions and the kernel becomes shared-memory bound (444 ms against
// 418 ms for two rows per lane on the 1000 vs 1000 x 2048 evaluation). So a lane keeps TWO rows (rows l and l + 16 of
// the leaf, l = lane & 15; lanes l and l ^ 16 hold the same rows) and half-warp h reads the candidate pairs 8 h .. 8 h + 7
// of the chunk -- an LDS.128 with one address per half-warp is still two wavefronts -- which halves the wavefronts per
// arithmetic instruction. Each lane tracks (minimum, runner-up, window) of both rows over ITS half of the candidates;
// the halves are merged with one shuffle per scanned chunk (pruning bound of the lane's own row: lane l + 16 h owns
// row l + 16 h) and three at the end of the walk.
// Shape, measured with 64-row groups on the same evaluation: 8 / 16 / 32 candidates per window 419 / 436 / 512 ms;
// 4 / 6 / 8 / 10 / 12 warps per CTA 466 / 435 / 418 / 416 / 415 ms (a plateau: bound by issue slots, not by latency).
constexpr int PAIR_CAP = 2048;
constexpr int PAIR_NW = 8;                 // warps per CTA

__global__ void __launch_bounds__(PAIR_NW * 32, 3) nn_pair_split_kernel(const Params p) {
  constexpr int SUB = 8;
  constexpr int GR = 32;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  __shared__ uint64_t bar;
  __shared__ double tsum[2 * (PAIR_CAP / GR)];
  __shared__ int next_task;
  const int tid = threadIdx.x, lane = tid & 31;
  const int h = lane >> 4, l16 = lane & 15;

  const int ci = p.row_begin + blockIdx.y * p.row_stride;
  const int cj = blockIdx.x;
  if (p.symmetric && cj < ci) return;

  const int2 mx = p.metaX[ci], my = p.metaY[cj];
  const int padX = (mx.x + CHUNK - 1) / CHUNK * CHUNK, padY = (my.x + CHUNK - 1) / CHUNK * CHUNK;
  float4* const sX = reinterpret_cast<float4*>(smem_raw);
  float4* const sY = sX + p.paddedX;
  float4* const bX = sY + p.paddedY;
  float4* const bY = bX + p.paddedX / CHUNK * 2;
  if (tid == 0) {
    mbar_init(&bar, 1);
    mbar_fence_init();
    next_task = 0;
    const uint32_t bytes = (uint32_t)(padX + padY) * 16u + (uint32_t)(padX / CHUNK + padY / CHUNK) * 32u;
    mbar_expect_tx(&bar, bytes);
    bulk_g2s(sX, p.scanX + (long long)ci * p.strideX, (uint32_t)padX * 16u, &bar);
    bulk_g2s(sY, p.scanY + (long long)cj * p.strideY, (uint32_t)padY * 16u, &bar);
    bulk_g2s(bX, p.boxX + (long long)ci * (p.paddedX / CHUNK * 2), (uint32_t)(padX / CHUNK) * 32u, &bar);
    bulk_g2s(bY, p.boxY + (long long)cj * (p.paddedY / CHUNK * 2), (uint32_t)(padY / CHUNK) * 32u, &bar);
  }
  __syncthreads();
  mbar_wait(&bar, 0);

  const int ngX = (mx.x + GR - 1) / GR, ngY = (my.x + GR - 1) / GR;
  const float inf = __int_as_float(0x7f800000);

  for (;;) {
    int task = 0;
    if (lane == 0) task = atomicAdd(&next_task, 1);
    task = __shfl_sync(0xffffffffu, task, 0);
    if (task >= ngX + ngY) break;
    const int dir = task >= ngX;
    const int g = dir ? task - ngX : task;
    const float4* const rows = dir ? sY : sX;
    const float4* const cand = dir ? sX : sY;
    const float4* const rbox = dir ? bY : bX;
    const float4* const cbox = dir ? bX : bY;
    const int rowcount = dir ? my.x : mx.x;
    const int nch = (dir ? padX : padY) / CHUNK;

    // ---- the lane's two rows (search operands), its OWN row (coordinates, bound), the leaf's box ----
    f32x2 nax[2], nay[2], naz[2];
    float cur[2], sec[2];
    int cid[2];
    float rx[2], ry[2], rz[2];
    #pragma unroll
    for (int j = 0; j < 2; ++j) {
      const int row = g * GR + j * 16 + l16;
      const int rr = row < rowcount ? row : 0;
      const float* f = reinterpret_cast<const float*>(rows + (rr >> 1) * 2) + (rr & 1);
      rx[j] = f[0]; ry[j] = f[2]; rz[j] = f[4];
      const float mx2 = -2.0f * rx[j], my2 = -2.0f * ry[j], mz2 = -2.0f * rz[j];
      nax[j] = pack2(mx2, mx2); nay[j] = pack2(my2, my2); naz[j] = pack2(mz2, mz2);
      cur[j] = sec[j] = inf; cid[j] = 0;
    }
    const float oax = h ? rx[1] : rx[0], oay = h ? ry[1] : ry[0], oaz = h ? rz[1] : rz[0];
    const float an = fmaf(oaz, oaz, fmaf(oax, oax, oay * oay));
    const int orow = g * GR + lane;                         // = g GR + 16 h + l16
    float ubr = orow < rowcount ? inf : -1.0f;              // a dead row never asks
    float gl0, gl1, gl2, gh0, gh1, gh2;
    {
      const float4 bl = rbox[2 * g], bh = rbox[2 * g + 1];
      gl0 = bl.x; gl1 = bl.y; gl2 = bl.z; gh0 = bh.x; gh1 = bh.y; gh2 = bh.z;
      if (bl.w != 0.0f) {          // the leaf also holds the merged origin point, kept outside its box
        gl0 = fminf(gl0, 0.0f); gl1 = fminf(gl1, 0.0f); gl2 = fminf(gl2, 0.0f);
        gh0 = fmaxf(gh0, 0.0f); gh1 = fmaxf(gh1, 0.0f); gh2 = fmaxf(gh2, 0.0f);
      }
    }
    const bool forced = cbox[2 * (nch - 1)].w != 0.0f;
    unsigned key[2];
    #pragma unroll
    for (int q = 0; q < 2; ++q) {
      const int c = q * 32 + lane;
      key[q] = 0xffffffffu;
      if (forced && c == nch - 1) {
        key[q] = (unsigned)c;
      } else if (c < nch) {
        const float4 bl = cbox[2 * c], bh = cbox[2 * c + 1];
        const float gx = max3(0.0f, bl.x - gh0, gl0 - bh.x), gy = max3(0.0f, bl.y - gh1, gl1 - bh.y), gz = max3(0.0f, bl.z - gh2, gl2 - bh.z);
        const float lb = fmaf(gz, gz, fmaf(gx, gx, __fmul_rn(gy, gy)));
        if (lb < inf) key[q] = (__float_as_uint(lb) & ~63u) | (unsigned)c;
      }
    }
    float ubmax = inf;
    int nvis = 0;
    for (;;) {
      const unsigned kwin = __reduce_min_sync(0xffffffffu, min(key[0], key[1]));
      if (kwin == 0xffffffffu) break;
      if (__uint_as_float(kwin & ~63u) > ubmax) break;
      const int c = (int)(kwin & 63u);
      if (key[0] == kwin) key[0] = 0xffffffffu;
      if (key[1] == kwin) key[1] = 0xffffffffu;
      const float4 bl = cbox[2 * c], bh = cbox[2 * c + 1];
      const float qx = max3(0.0f, bl.x - oax, oax - bh.x), qy = max3(0.0f, bl.y - oay, oay - bh.y), qz = max3(0.0f, bl.z - oaz, oaz - bh.z);
      const bool need = (forced && c == nch - 1) || fmaf(qz, qz, fmaf(qx, qx, __fmul_rn(qy, qy))) <= ubr;
      if (!__any_sync(0xffffffffu, need)) continue;
      ++nvis;
      const float4* cp = cand + c * CHUNK + h * (CHUNK / 2);      // this half-warp's 16 candidates
      #pragma unroll
      for (int w = 0; w < 2; ++w) {
        float cm[2];
        #pragma unroll
        for (int k = w * 4; k < w * 4 + 4; ++k) {
          const float4 q0 = cp[2 * k], q1 = cp[2 * k + 1];
          const f32x2 bx = pack2(q0.x, q0.y), by = pack2(q0.z, q0.w);
          const f32x2 bz = pack2(q1.x, q1.y), bn = pack2(q1.z, q1.w);
          #pragma unroll
          for (int j = 0; j < 2; ++j) {
            f32x2 s = fma2(naz[j], bz, bn);
            s = fma2(nay[j], by, s);
            s = fma2(nax[j], bx, s);
            float lo, hi;
            unpack2(s, lo, hi);
            cm[j] = (k == w * 4) ? fminf(lo, hi) : min3(cm[j], lo, hi);
          }
        }
        const int wid = c * (CHUNK / SUB) + 2 * h + w;
        #pragma unroll
        for (int j = 0; j < 2; ++j) {
          const bool better = cm[j] < cur[j];
          sec[j] = fminf(sec[j], better ? cur[j] : cm[j]);      // (an all-padding window has cm = NaN: ignored)
          cur[j] = fminf(cur[j], cm[j]);
          cid[j] = better ? wid : cid[j];
        }
      }
      // bound of the lane's own row from both halves' minima (the partner sends its minimum for the row it does not own)
      const float other = __shfl_xor_sync(0xffffffffu, h ? cur[0] : cur[1], 16);
      if (ubr >= 0.0f) {
        const float dest = fmaxf(fminf(h ? cur[1] : cur[0], other) + an, 0.0f);
        ubr = fmaf(3.81469727e-6f /* 64 * 2^-24 */, an + dest, dest) + 1e-36f;
      }
      ubmax = __uint_as_float(__reduce_max_sync(0xffffffffu, __float_as_uint(fmaxf(ubr, 0.0f))));
    }
    if (p.visited != nullptr && lane == 0)
      atomicAdd(p.visited, (unsigned long long)nvis * CHUNK * (unsigned long long)min(GR, rowcount - g * GR));

    // ---- merge the halves, exact pass on the own row's winning window, guard over the whole candidate cloud ----
    const float pc = __shfl_xor_sync(0xffffffffu, h ? cur[0] : cur[1], 16);
    const float ps = __shfl_xor_sync(0xffffffffu, h ? sec[0] : sec[1], 16);
    const int pi = __shfl_xor_sync(0xffffffffu, h ? cid[0] : cid[1], 16);
    const float mc = h ? cur[1] : cur[0], ms = h ? sec[1] : sec[0];
    const int mi0 = h ? cid[1] : cid[0];
    const bool theirs = pc < mc;
    const float c1 = fminf(mc, pc);
    const float s1 = fminf(fminf(ms, ps), theirs ? mc : pc);      // the halves' windows are disjoint
    const int w1 = theirs ? pi : mi0;
    const bool live = orow < rowcount;
    float e = inf;
    if (live && c1 < inf) {
      const f32x2 ax2 = pack2(oax, oax), ay2 = pack2(oay, oay), az2 = pack2(oaz, oaz);
      const float4* cp = cand + w1 * SUB;
      #pragma unroll
      for (int k = 0; k < SUB / 2; ++k) {
        const int kk = (k + lane) & (SUB / 2 - 1);      // lanes start on different banks
        const float4 q0 = cp[2 * kk], q1 = cp[2 * kk + 1];
        const f32x2 dx = sub2(pack2(q0.x, q0.y), ax2);
        const f32x2 dy = sub2(pack2(q0.z, q0.w), ay2);
        const f32x2 dz = sub2(pack2(q1.x, q1.y), az2);
        float lo, hi;
        unpack2(fma2(dz, dz, fma2(dx, dx, mul2(dy, dy))), lo, hi);
        e = min3(e, lo, hi);
      }
    }
    const bool near_tie = live && s1 <= c1 + search_window(oax, oay, oaz, c1);
    unsigned flagged = __ballot_sync(0xffffffffu, near_tie);
    while (flagged) {                         // warp-uniform
      const int src = __ffs(flagged) - 1;
      flagged &= flagged - 1;
      float m;
      int mi;
      warp_cloud_exact_min<false>(cand, nch, cbox, __shfl_sync(0xffffffffu, e, src), __shfl_sync(0xffffffffu, oax, src),
                                  __shfl_sync(0xffffffffu, oay, src), __shfl_sync(0xffffffffu, oaz, src), lane, nullptr, m, mi);
      if (lane == src) e = fminf(e, m);
    }
    double dsum = live ? (orow == rowcount - 1 ? (double)(dir ? my.y : mx.y) : 1.0) * (double)e : 0.0;
    #pragma unroll
    for (int o = 16; o > 0; o >>= 1) dsum += __shfl_down_sync(0xffffffffu, dsum, o);
    if (lane == 0) tsum[task] = dsum;
  }

  __syncthreads();
  if (tid == 0) {
    double S0 = 0.0, S1 = 0.0;
    for (int t = 0; t < ngX; ++t) S0 += tsum[t];
    for (int t = ngX; t < ngX + ngY; ++t) S1 += tsum[t];
    emit_entry(p, ci, cj, S0, S1);
  }
}

static int launch_pair_split(const Params& p, dim3 grid, cudaStream_t st) {
  const size_t smem = (size_t)(p.paddedX + p.paddedY) * 16 + (size_t)(p.paddedX / CHUNK + p.paddedY / CHUNK) * 32;
  static bool configured[kMaxDevices] = {};
  const int dev = current_device();
  if (!configured[dev]) {
    DUSTY_CUDA(cudaFuncSetAttribute(nn_pair_split_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    2 * PAIR_CAP * 16 + 2 * (PAIR_CAP / CHUNK) * 32));
    configured[dev] = true;
  }
  nn_pair_split_kernel<<<grid, PAIR_NW * 32, smem, st>>>(p);
  DUSTY_AFTER_LAUNCH("chamfer nn_pair_split_kernel");
  return 0;
}
