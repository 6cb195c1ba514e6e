// Best-first Chamfer search for sorted clouds of any size up to SORT_CAP (un-sampled range images: configs[4],
// compute_cd on reconstruction pairs): included by chamfer.cu inside namespace dusty::chamfer.
//
// The walk of nn_pair_split_kernel (chamfer_pair.cuh) -- 32-row groups, two rows per lane, the two half-warps on the two
// halves of a candidate chunk, lane l + 16 h owns row l + 16 h -- with two changes for clouds that do not fit shared memory:
//   * two levels: a lane first bounds one BLOCK of 32 chunks (1024 consecutive points of the candidate cloud, a subtree
//     of its k-d tree in k-d order; at most 32 blocks, their boxes come from prep_sort_kernel) and the warp opens blocks
//     best first; inside an open block a lane bounds one chunk and the warp scans chunks best first. Both levels stop
//     at the first bound beyond the largest running minimum of the warp's 32 rows;
//   * candidates, boxes and rows are read from global memory through L1 (the kernel uses little shared memory, so L1
//     keeps ~200 KB): row groups are taken in sorted order, so the warps of a CTA work on neighbouring groups and walk
//     overlapping chunks. The chunk a warp scans is staged through 512 bytes of per-warp shared memory: a
//     half-warp-uniform LDG.128 costs far more L1 wavefronts than the same LDS.128.
// The walk reads only the chunks it scans -- on the bench's un-sampled clouds 1.7 % of the kept pairs (64-row groups:
// 2.3 %) -- where streaming every tile of the candidate cloud past every row block moves 33 MB from L2 to shared memory
// per entry at 16 k points.
// MATRIX: one CTA per matrix entry, per-task sums added in task order (deterministic under the dynamic task
// order). Batch front end (Morton order): a CTA takes WALK_TPC consecutive tasks of one pair; per-point (dist, idx) go to
// the sorted positions and unsort_kernel puts them back (ties between bit-equal distances: lowest original index, through
// perm).
constexpr int WALK_NW = 8;                  // warps per CTA
constexpr int WALK_TPC = 8;                 // tasks per CTA in the batch front end (one per warp: few pairs must still fill the GPU)
constexpr int WALK_SPLIT_MAXTASKS = 2 * (SORT_CAP / 32 + 1);

template <bool MATRIX>
__global__ void __launch_bounds__(WALK_NW * 32, 3) nn_walk_split_kernel(const Params p) {
  constexpr int SUB = 8;
  constexpr int GR = 32;
  __shared__ double tsum[MATRIX ? WALK_SPLIT_MAXTASKS : 1];
  __shared__ int next_task;
  __shared__ float4 stage[WALK_NW][CHUNK];      // the chunk a warp scans: one coalesced 512-byte load instead of 16 half-warp-uniform ones
  const int tid = threadIdx.x, lane = tid & 31;
  const int h = lane >> 4, l16 = lane & 15;
  int ci, cj;
  if (MATRIX) {
    ci = p.row_begin + blockIdx.y * p.row_stride;
    cj = blockIdx.x;
    if (p.symmetric && cj < ci) return;
  } else {
    ci = cj = blockIdx.y;
  }
  const int2 mx = p.metaX[ci], my = p.metaY[cj];
  const int padX = (mx.x + CHUNK - 1) / CHUNK * CHUNK, padY = (my.x + CHUNK - 1) / CHUNK * CHUNK;
  const float4* const sX = p.scanX + (long long)ci * p.strideX;
  const float4* const sY = p.scanY + (long long)cj * p.strideY;
  const float4* const bX = p.boxX + (long long)ci * (p.paddedX / CHUNK * 2);
  const float4* const bY = p.boxY + (long long)cj * (p.paddedY / CHUNK * 2);
  const float4* const bbX = p.bbX + (long long)ci * (2 * WALK_BLOCKS);
  const float4* const bbY = p.bbY + (long long)cj * (2 * WALK_BLOCKS);

  const int ngX = (mx.x + GR - 1) / GR, ngY = (my.x + GR - 1) / GR;
  int task_begin = 0, task_end = ngX + ngY;
  if (!MATRIX) {
    task_begin = blockIdx.x * WALK_TPC;
    task_end = min(task_end, task_begin + WALK_TPC);
    if (task_begin >= task_end) return;
  }
  if (tid == 0) next_task = task_begin;
  __syncthreads();
  const float inf = __int_as_float(0x7f800000);

  for (;;) {
    int task = 0;
    if (lane == 0) task = atomicAdd(&next_task, 1);
    task = __shfl_sync(0xffffffffu, task, 0);
    if (task >= task_end) break;
    const int dir = task >= ngX;
    const int g = dir ? task - ngX : task;
    const float4* const rows = dir ? sY : sX;
    const float4* const cand = dir ? sX : sY;
    const float4* const rbox = dir ? bY : bX;
    const float4* const cbox = dir ? bX : bY;
    const float4* const cblk = dir ? bbX : bbY;
    const int* const cperm = MATRIX ? nullptr : (dir ? p.permX + (long long)ci * p.strideX : p.permY + (long long)cj * p.strideY);
    const int rowcount = dir ? my.x : mx.x;
    const int nch = (dir ? padX : padY) / CHUNK;
    const int nblk = (nch + 31) / 32;

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
    const int orow = g * GR + lane;
    float ubr = orow < rowcount ? inf : -1.0f;
    float gl0, gl1, gl2, gh0, gh1, gh2;
    {
      const float4 bl = rbox[2 * g], bh = rbox[2 * g + 1];
      gl0 = bl.x; gl1 = bl.y; gl2 = bl.z; gh0 = bh.x; gh1 = bh.y; gh2 = bh.z;
      if (bl.w != 0.0f) {          // the leaf also holds the merged origin point, kept outside its box
        gl0 = fminf(gl0, 0.0f); gl1 = fminf(gl1, 0.0f); gl2 = fminf(gl2, 0.0f);
        gh0 = fmaxf(gh0, 0.0f); gh1 = fmaxf(gh1, 0.0f); gh2 = fmaxf(gh2, 0.0f);
      }
    }
    auto box_key = [&](const float4& bl, const float4& bh, unsigned id) -> unsigned {
      const float gx = max3(0.0f, bl.x - gh0, gl0 - bh.x), gy = max3(0.0f, bl.y - gh1, gl1 - bh.y), gz = max3(0.0f, bl.z - gh2, gl2 - bh.z);
      const float lb = fmaf(gz, gz, fmaf(gx, gx, __fmul_rn(gy, gy)));
      return lb < inf ? (__float_as_uint(lb) & ~31u) | id : 0xffffffffu;
    };
    const bool forced = cbox[2 * (nch - 1)].w != 0.0f;
    unsigned bkey = 0xffffffffu;
    if (lane < nblk) bkey = forced && lane == nblk - 1 ? (unsigned)lane : box_key(cblk[2 * lane], cblk[2 * lane + 1], (unsigned)lane);
    float ubmax = inf;
    int nvis = 0;
    for (;;) {
      const unsigned bwin = __reduce_min_sync(0xffffffffu, bkey);
      if (bwin == 0xffffffffu || __uint_as_float(bwin & ~31u) > ubmax) break;
      const int blk = (int)(bwin & 31u);
      if (bkey == bwin) bkey = 0xffffffffu;
      unsigned key = 0xffffffffu;
      const int cl = blk * 32 + lane;
      if (cl < nch) key = forced && cl == nch - 1 ? (unsigned)lane : box_key(cbox[2 * cl], cbox[2 * cl + 1], (unsigned)lane);
      for (;;) {
        const unsigned kwin = __reduce_min_sync(0xffffffffu, key);
        if (kwin == 0xffffffffu || __uint_as_float(kwin & ~31u) > ubmax) break;
        const int c = blk * 32 + (int)(kwin & 31u);
        if (key == kwin) key = 0xffffffffu;
        const float4 bl = cbox[2 * c], bh = cbox[2 * c + 1];
        const float qx = max3(0.0f, bl.x - oax, oax - bh.x), qy = max3(0.0f, bl.y - oay, oay - bh.y), qz = max3(0.0f, bl.z - oaz, oaz - bh.z);
        const bool need = (forced && c == nch - 1) || fmaf(qz, qz, fmaf(qx, qx, __fmul_rn(qy, qy))) <= ubr;
        if (!__any_sync(0xffffffffu, need)) continue;
        ++nvis;
        __syncwarp();                          // everyone is done with the previous chunk
        stage[tid >> 5][lane] = __ldg(cand + (long long)c * CHUNK + lane);
        __syncwarp();
        const float4* cp = &stage[tid >> 5][h * (CHUNK / 2)];      // this half-warp's 16 candidates
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
        const float other = __shfl_xor_sync(0xffffffffu, h ? cur[0] : cur[1], 16);
        if (ubr >= 0.0f) {
          const float dest = fmaxf(fminf(h ? cur[1] : cur[0], other) + an, 0.0f);
          ubr = fmaf(3.81469727e-6f /* 64 * 2^-24 */, an + dest, dest) + 1e-36f;
        }
        ubmax = __uint_as_float(__reduce_max_sync(0xffffffffu, __float_as_uint(fmaxf(ubr, 0.0f))));
      }
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
    const float s1 = fminf(fminf(ms, ps), theirs ? mc : pc);
    const int w1 = theirs ? pi : mi0;
    const bool live = orow < rowcount;
    float e = inf;
    int eidx = 0x7fffffff;
    if (live && c1 < inf) {
      const f32x2 ax2 = pack2(oax, oax), ay2 = pack2(oay, oay), az2 = pack2(oaz, oaz);
      const float4* cp = cand + (long long)w1 * SUB;
      #pragma unroll
      for (int k = 0; k < SUB / 2; ++k) {
        const float4 q0 = __ldg(cp + 2 * k), q1 = __ldg(cp + 2 * k + 1);
        const f32x2 dx = sub2(pack2(q0.x, q0.y), ax2);
        const f32x2 dy = sub2(pack2(q0.z, q0.w), ay2);
        const f32x2 dz = sub2(pack2(q1.x, q1.y), az2);
        float lo, hi;
        unpack2(fma2(dz, dz, fma2(dx, dx, mul2(dy, dy))), lo, hi);
        if (MATRIX) {
          e = min3(e, lo, hi);
        } else {
          const int i0 = w1 * SUB + 2 * k;
          if (lo < e || (lo == e && eidx != 0x7fffffff && cperm[i0] < cperm[eidx])) { e = lo; eidx = i0; }
          if (hi < e || (hi == e && eidx != 0x7fffffff && cperm[i0 + 1] < cperm[eidx])) { e = hi; eidx = i0 + 1; }
        }
      }
    }
    const bool near_tie = live && s1 <= c1 + search_window(oax, oay, oaz, c1);
    unsigned flagged = __ballot_sync(0xffffffffu, near_tie);
    while (flagged) {                         // warp-uniform
      const int src = __ffs(flagged) - 1;
      flagged &= flagged - 1;
      float m;
      int mi = 0x7fffffff;
      warp_cloud_exact_min<!MATRIX>(cand, nch, cbox, __shfl_sync(0xffffffffu, e, src), __shfl_sync(0xffffffffu, oax, src),
                                    __shfl_sync(0xffffffffu, oay, src), __shfl_sync(0xffffffffu, oaz, src), lane, cperm, m, mi);
      if (lane == src) {
        if (MATRIX) {
          e = fminf(e, m);
        } else if (mi != 0x7fffffff && (m < e || (m == e && (eidx == 0x7fffffff || cperm[mi] < cperm[eidx])))) {
          e = m; eidx = mi;
        }
      }
    }
    if (MATRIX) {
      double dsum = live ? (orow == rowcount - 1 ? (double)(dir ? my.y : mx.y) : 1.0) * (double)e : 0.0;
      #pragma unroll
      for (int o = 16; o > 0; o >>= 1) dsum += __shfl_down_sync(0xffffffffu, dsum, o);
      if (lane == 0) tsum[task] = dsum;
    } else if (live) {            // per sorted position (stride = padded count); unsort_kernel restores the original order
      const long long o = (long long)ci * (dir ? p.strideY : p.strideX) + orow;
      (dir ? p.dist2 : p.dist1)[o] = e;
      (dir ? p.idx2 : p.idx1)[o] = cperm[eidx == 0x7fffffff ? 0 : eidx];
    }
  }

  if (MATRIX) {
    __syncthreads();
    if (tid == 0) {
      double S0 = 0.0, S1 = 0.0;
      for (int t = 0; t < ngX; ++t) S0 += tsum[t];
      for (int t = ngX; t < ngX + ngY; ++t) S1 += tsum[t];
      emit_entry(p, ci, cj, S0, S1);
    }
  }
}

template <bool MATRIX>
static int launch_walk_split(const Params& p, dim3 grid, cudaStream_t st) {
  nn_walk_split_kernel<MATRIX><<<grid, WALK_NW * 32, 0, st>>>(p);
  DUSTY_AFTER_LAUNCH("chamfer nn_walk_split_kernel");
  return 0;
}
