/*
 * dusty_b200.h -- C ABI of libdustyb200.so: the B200 (sm_100a) kernels behind DUSty-GAN's
 * generate-and-evaluate hot path.
 *
 * This is the drop-in boundary. Every entry point takes plain device pointers, sizes and a CUDA
 * stream (passed as void* so that the header needs no CUDA include); none allocates memory and none
 * keeps state between calls. Scratch space is supplied by the caller; each function that needs it
 * has a matching *_workspace_bytes() query. Every function returns 0 on success, a positive
 * cudaError_t value when the CUDA runtime reported an error, or a negative DUSTY_E* value for an
 * argument error. dusty_last_error_string() describes the last non-zero return on this thread.
 *
 * Reference interfaces replaced (paths are relative to the kazuto1011/dusty-gan tree):
 *   dusty_chamfer_forward        utils/metrics/distance/cd/chamfer_distance.cpp:16-25  (cd.forward_cuda)
 *                                -> ChamferDistanceKernelLauncher, chamfer_distance.cu:133-146
 *   dusty_chamfer_backward       utils/metrics/distance/cd/chamfer_distance.cpp:27-37  (cd.backward_cuda)
 *                                -> ChamferDistanceGradKernelLauncher, chamfer_distance.cu:174-190
 *   dusty_chamfer_matrix         utils/metrics/cov_mmd_1nna.py:24-51 (_pairwise_distance, the Python
 *                                double loop over compute_cd, :19-21)
 *   dusty_cov_mmd_1nna_finalize  utils/metrics/cov_mmd_1nna.py:54-106 (_compute_cov_mmd, _compute_nna k=1)
 *   dusty_chamfer_matrix_fused, dusty_nn_keys_*, dusty_cov_mmd_1nna_from_keys
 *                                utils/metrics/cov_mmd_1nna.py:109-139 (compute_cov_mmd_1nna): the three
 *                                _pairwise_distance calls with the min / arg-min / topk reductions of :54-106
 *                                folded into the matrix kernel's epilogue -- no (Nr+Ng)^2 tensor is ever stored
 *   dusty_symmetric_from_shards  the multi-GPU assembly of a row-sharded symmetric matrix (no reference
 *                                counterpart: the reference is single-GPU on this path)
 *   dusty_emd_forward            utils/metrics/distance/emd/ (approxmatch + matchcost, SURVEY.md S2a), the
 *                                forward of earth_mover_distance; no (b,m,n) match matrix
 *   dusty_emd_backward           the same extension's matchcostgrad1 / matchcostgrad2
 *   dusty_emd_matrix             utils/metrics/cov_mmd_1nna.py compute_emd and the "emd" metric of
 *                                compute_cov_mmd_1nna, with the fused minima of dusty_chamfer_matrix_fused
 *   dusty_jsd_vote, dusty_jsd_from_counts   utils/metrics/jsd.py:23-92, 110-121 (entropy_of_occupancy_grid,
 *                                _jensen_shannon_divergence)
 *   dusty_fps                    utils/sampling/fps/furthest_point_sampling.cpp:79-100
 *                                -> furthest_point_sampling_kernel_wrapper, furthest_point_sampling.cu:209-260
 *   dusty_gather_points          utils/sampling/fps/furthest_point_sampling.cpp:27-50
 *                                -> gather_points_kernel_wrapper, furthest_point_sampling.cu:52-60
 *   dusty_gather_points_grad     utils/sampling/fps/furthest_point_sampling.cpp:52-77
 *   dusty_logistic_noise         models/dusty.py:30-36   (GumbelSigmoid.logistic_noise, given U1,U2)
 *   dusty_gumbel_sigmoid         models/dusty.py:38-59   (sigmoid_with_temperature + GumbelSigmoid.forward)
 *   dusty_head_project           models/dusty.py:45-59,77-91,107-127 (GumbelSigmoid.forward,
 *                                DUSty1.maskout, DUSty2.maskout) fused with utils/__init__.py:76-79
 *                                (tanh_to_sigmoid + clamp) and utils/lidar.py:38-68 (inv_to_xyz)
 *   dusty_head_project_backward  the autograd backward of the same chain (the straight-through mask gradient),
 *                                e.g. demo.py:510-515's inversion loss and the generator step of trainers/dcgan_amp.py
 *   dusty_inv_to_xyz             utils/lidar.py:61-68     (Coordinate.inv_to_xyz alone)
 *   dusty_scan_preprocess        datasets/kitti.py:54-78 (KITTIOdometry.preprocess + transform's nearest
 *                                resize) fused with evaluate_synthesis.py:49-57 (preprocess_reals:
 *                                utils/lidar.py:31-36 invert_depth, utils/__init__.py:70-73 sigmoid_to_tanh,
 *                                mask blend, flatten/transpose): the real-data side of the path
 */
#ifndef DUSTY_B200_H_
#define DUSTY_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DUSTY_B200_ABI_VERSION 3

#if defined(__GNUC__)
#define DUSTY_API __attribute__((visibility("default")))
#else
#define DUSTY_API
#endif

/* negative return codes (argument errors); positive codes are cudaError_t values */
#define DUSTY_EINVAL   (-1)   /* bad size / flag / null pointer */
#define DUSTY_EALIGN   (-2)   /* pointer not aligned as documented */
#define DUSTY_ENOSPACE (-3)   /* workspace smaller than *_workspace_bytes() */
#define DUSTY_EARCH    (-4)   /* device is not compute capability 10.x */

DUSTY_API int dusty_abi_version(void);
DUSTY_API const char* dusty_last_error_string(void);
/* Number of kernels this library has launched in this process (all streams); bench.py reads it
 * before and after the timed region to report gpu_launches. */
DUSTY_API uint64_t dusty_launch_count(void);

/* --------------------------------------------------------------------------------------------
 * Chamfer nearest-neighbour search
 * -------------------------------------------------------------------------------------------- */

/* Scratch for dusty_chamfer_forward on (b,n,3) x (b,m,3). */
DUSTY_API size_t dusty_chamfer_forward_workspace_bytes(int b, int n, int m);

/* Directed nearest neighbours in both directions for b independent cloud pairs.
 *   xyz1 (b,n,3) f32, xyz2 (b,m,3) f32, contiguous.
 *   dist1 (b,n) f32: min_k |xyz1[i,j]-xyz2[i,k]|^2 evaluated as fma(dz,dz,fma(dx,dx,dy*dy)), the
 *   rounding pattern of the reference kernel; idx1 (b,n) i32 the arg-min (lowest index among
 *   bit-equal candidates). dist2/idx2 likewise for xyz2 against xyz1. idx1/idx2 may be NULL.
 *   When n == 0 or m == 0 the outputs are zero-filled, as the reference leaves them. */
DUSTY_API int dusty_chamfer_forward(const float* xyz1, const float* xyz2, int b, int n, int m,
                          float* dist1, float* dist2, int32_t* idx1, int32_t* idx2,
                          void* workspace, size_t workspace_bytes, void* stream);

/* Gradient of sum(grad_dist1*dist1)+sum(grad_dist2*dist2) w.r.t. both clouds, given the forward
 * arg-mins. grad_xyz1 (b,n,3) and grad_xyz2 (b,m,3) are overwritten: every element is first written with
 * its own term 2 g (p - q) (no memset, no atomic), then the neighbour terms of both directions are added
 * with atomicAdd (warp-aggregated per target), so -- as in the reference kernel -- the summation order of
 * colliding targets is not fixed. */
DUSTY_API size_t dusty_chamfer_backward_workspace_bytes(int b, int n, int m);
DUSTY_API int dusty_chamfer_backward(const float* xyz1, const float* xyz2, int b, int n, int m,
                           const float* grad_dist1, const float* grad_dist2,
                           const int32_t* idx1, const int32_t* idx2,
                           float* grad_xyz1, float* grad_xyz2,
                           void* workspace, size_t workspace_bytes, void* stream);

/* Scratch for dusty_chamfer_matrix over na + nb clouds (nb = 0 when symmetric). */
DUSTY_API size_t dusty_chamfer_matrix_workspace_bytes(int na, int pa, int nb, int pb);

/* Pairwise Chamfer matrix between two sets of clouds:
 *   M[i,j] = mean_p min_q |A[i,p]-B[j,q]|^2 + mean_q min_p |A[i,p]-B[j,q]|^2     (compute_cd)
 *   A (na,pa,3) f32, B (nb,pb,3) f32, M row-major with leading dimension ldm (>= nb), f32.
 *   Only rows i = row_begin, row_begin + row_stride, ... < row_end are computed (the multi-GPU row
 *   shard; a stride equal to the number of ranks balances the triangular case); other rows of M
 *   are not touched.
 *   flags:
 *     DUSTY_MATRIX_SYMMETRIC     B is A (same pointer, nb == na, pb == pa): only entries with j >= i
 *                                of the owned rows are computed;
 *     DUSTY_MATRIX_MIRROR        with SYMMETRIC, also store each entry at M[j,i] (bit-equal in the
 *                                reference because float addition commutes);
 *     DUSTY_MATRIX_COMPACT_ROWS  store owned row number r (0,1,2,...) at M[r,:] instead of M[i,:],
 *                                i.e. M is the rank's (rows_owned, nb) block ready for an all-gather
 *                                (incompatible with MIRROR);
 *     DUSTY_MATRIX_PREPARED      the workspace already holds the scan-format copies of these A,B
 *                                from an earlier call (with the same MERGE_ORIGIN choice): skip
 *                                rebuilding them;
 *     DUSTY_MATRIX_MERGE_ORIGIN  un-sampled clouds keep every dropped pixel as a (0,0,0) point
 *                                (evaluate_reconstruction.py:124-131, SURVEY.md S7). All exactly-zero
 *                                points of a cloud are scanned as ONE point of that multiplicity:
 *                                the minima are unchanged (duplicate candidates never change a
 *                                minimum, identical rows share theirs) and the means still divide
 *                                by pa / pb, so M is the same matrix for a fraction of the work.
 *                                Clouds of at most 32768 points are also put in spatial (k-d) order
 *                                with a bounding box per 32 points, and the kernel walks candidate
 *                                chunks best first by box distance, skipping every chunk whose box is
 *                                no closer to a warp's rows than their current minima -- exact, the
 *                                bound is evaluated in the kernel's own rounding. Clouds of at most 2048
 *                                points are searched from shared memory (both clouds resident). */
#define DUSTY_MATRIX_SYMMETRIC    1
#define DUSTY_MATRIX_MIRROR       2
#define DUSTY_MATRIX_COMPACT_ROWS 4
#define DUSTY_MATRIX_PREPARED     8
#define DUSTY_MATRIX_MERGE_ORIGIN 16
DUSTY_API int dusty_chamfer_matrix(const float* A, int na, int pa, const float* B, int nb, int pb,
                         int row_begin, int row_end, int row_stride, int flags,
                         float* M, long long ldm,
                         void* workspace, size_t workspace_bytes, void* stream);

/* Fused evaluation (compute_cov_mmd_1nna, reference cov_mmd_1nna.py:109-139): the same launch as
 * dusty_chamfer_matrix, and every computed entry (i, j) also feeds the reductions _compute_cov_mmd and
 * _compute_nna(k = 1) need, as 64-bit atomic minima of (float bits of M[i,j] << 32 | stacked index):
 *   keys[0*n_total + c]  nearest other cloud of stacked cloud c (the +inf diagonal of :82 is skipped);
 *   keys[1*n_total + c]  for a generated cloud c: its nearest reference cloud   (MMD-sample, COV);
 *   keys[2*n_total + c]  for a reference cloud c: its nearest generated cloud   (MMD).
 * "Stacked" is the order of _compute_nna's matrix: the n_ref reference clouds first, then the generated
 * ones; cloud i of A is stacked cloud stacked_offset_a + i, cloud j of B is stacked_offset_b + j. Every
 * unordered pair of stacked clouds must be computed by exactly one launch / row shard (one symmetric launch
 * over the stacked set, or M_rr, M_rg, M_gg as three launches). Ties resolve to the lowest stacked index.
 * M may be NULL: then the matrix is not stored at all -- peak memory is O(n_total), not O(n_total^2).
 * keys (3*n_total u64) must be reset with dusty_nn_keys_reset before the first launch of an evaluation.
 * Across GPUs every rank fills its own key set from its row shard; the sets are all-gathered (24*n_total
 * bytes per rank) and dusty_cov_mmd_1nna_from_keys reduces over them. */
DUSTY_API size_t dusty_nn_keys_bytes(int n_total);
DUSTY_API int dusty_nn_keys_reset(uint64_t* keys, int n_total, void* stream);
DUSTY_API int dusty_chamfer_matrix_fused(const float* A, int na, int pa, const float* B, int nb, int pb,
                         int row_begin, int row_end, int row_stride, int flags,
                         float* M, long long ldm,
                         int stacked_offset_a, int stacked_offset_b, int n_ref, int n_total, uint64_t* keys,
                         void* workspace, size_t workspace_bytes, void* stream);
/* out7 as dusty_cov_mmd_1nna_finalize, from `shards` gathered key sets (shards * 3 * (nr+ng) u64, set s at
 * keys + s*3*(nr+ng)); workspace: dusty_cov_mmd_1nna_workspace_bytes(nr, ng). */
DUSTY_API int dusty_cov_mmd_1nna_from_keys(const uint64_t* keys, int shards, int nr, int ng, float* out7,
                                 void* workspace, size_t workspace_bytes, void* stream);

/* Full symmetric (n,n) matrix from the gathered compact row blocks of a cyclic row deal: blocks (shards, cap, n),
 * block g row r = global row g + r*shards, entries j >= i valid (DUSTY_MATRIX_SYMMETRIC | COMPACT_ROWS). Every
 * entry of out is read from the shard that computed it (M[i,j] for i > j comes from M[j,i]: bit-equal in the
 * reference, SURVEY.md S8). n <= 65535. */
DUSTY_API int dusty_symmetric_from_shards(const float* blocks, int shards, int cap, int n, float* out, long long ldo,
                                void* stream);

/* MMD / COV / 1-NNA from the three matrices, on the device (no host round trip).
 *   Mrr (nr,nr), Mrg (nr,ng), Mgg (ng,ng) row-major f32, contiguous.
 *   out[0..6] (f32): mmd (mean_i min_j Mrg), mmd-sample (mean_j min_i Mrg), the NUMBER of distinct
 *   arg-min_i over the columns (COV = that / nr, divided by the caller in double like the
 *   reference), tp, fp, fn, tn of the leave-one-out 1-NN classifier (label ref = 1) on the
 *   stacked (nr+ng)^2 matrix with +inf diagonal; ties resolve to the lowest stacked index. */
DUSTY_API size_t dusty_cov_mmd_1nna_workspace_bytes(int nr, int ng);
DUSTY_API int dusty_cov_mmd_1nna_finalize(const float* Mrr, const float* Mrg, const float* Mgg, int nr, int ng,
                                float* out7, void* workspace, size_t workspace_bytes, void* stream);
/* The same with a k-nearest-neighbour vote, 1 <= k <= 64 (_compute_nna(k), cov_mmd_1nna.py:84-90): tp/fp/fn/tn come
 * from pred = (#reference clouds among the k nearest) / k >= 0.5; mmd, mmd-sample and the COV count are unchanged.
 * The reference's optional sqrt of the distances is monotone and does not change the neighbour sets. */
DUSTY_API int dusty_cov_mmd_knna_finalize(const float* Mrr, const float* Mrg, const float* Mgg, int nr, int ng, int k,
                                float* out7, void* workspace, size_t workspace_bytes, void* stream);

/* --------------------------------------------------------------------------------------------
 * Approximate Earth Mover's Distance (reference utils/metrics/distance/emd/: the PSGN approxmatch)
 * -------------------------------------------------------------------------------------------- */

/* Scratch for dusty_emd_forward on (b,n,3) x (b,m,3). */
DUSTY_API size_t dusty_emd_forward_workspace_bytes(int b, int n, int m);

/* Approximate EMD of b independent cloud pairs, bit-equal to the reference's approxmatch + matchcost kernels.
 *   xyz1 (b,n,3) f32, xyz2 (b,m,3) f32, contiguous; n, m >= 1.
 *   cost (b) f32: sum_{k,l} |xyz1[k] - xyz2[l]| match[l][k] (not divided by the point count).
 *   factors (b,10,n+m) f32 or NULL: the ten per-level ratio vectors (level v = 7 - j: ratioL (n), then
 *   ratioR (m)) from which dusty_emd_backward rebuilds the match. No (b,m,n) match matrix is stored. */
DUSTY_API int dusty_emd_forward(const float* xyz1, const float* xyz2, int b, int n, int m, float* cost,
                                float* factors, void* workspace, size_t workspace_bytes, void* stream);

/* Gradient of sum(grad_cost * cost) with the match held constant (the reference's matchcostgrad1/2):
 *   grad1[k] = grad_cost * sum_l match[l][k] (xyz1[k] - xyz2[l]) / max(|xyz1[k] - xyz2[l]|, 1e-20), grad2 the same
 *   with the sign flipped. factors from dusty_emd_forward on the same clouds. grad1 (b,n,3) and grad2 (b,m,3) are
 *   overwritten. No scratch is needed: workspace may be NULL. */
DUSTY_API int dusty_emd_backward(const float* xyz1, const float* xyz2, int b, int n, int m, const float* grad_cost,
                                 const float* factors, float* grad1, float* grad2,
                                 void* workspace, size_t workspace_bytes, void* stream);

/* Scratch for dusty_emd_matrix on A (na,pa,3) x B (nb,pb,3). */
DUSTY_API size_t dusty_emd_matrix_workspace_bytes(int na, int pa, int nb, int pb);

/* Pairwise EMD matrix (compute_emd of cov_mmd_1nna.py, each entry bit-equal to the one-pair forward):
 *   M[i,j] = cost(A[i], B[j]) * f32(1/pa), for rows i = row_begin, row_begin + row_stride, ... < row_end; M
 *   row-major with leading dimension ldm (>= nb), NULL: not stored. EMD is not symmetric: every entry is computed.
 * With keys (3*n_total u64, reset by dusty_nn_keys_reset) every entry also feeds the packed minima of
 * dusty_chamfer_matrix_fused, so dusty_cov_mmd_1nna_from_keys gives the scores. Cloud i of A is stacked cloud
 * stacked_offset_a + i, cloud j of B stacked_offset_b + j (reference clouds first). The 1-NN matrix
 * [[M_rr, M_rg], [M_rg^T, M_gg]] is reduced column-wise (topk(dim=0)): entry (r, c) feeds keys[c] with index r when
 * r != c; an M_rg entry (r < n_ref <= c) also feeds keys[r] with c, keys[n_total + c] with r and
 * keys[2 n_total + r] with c. A launch is reference-by-reference, reference-by-generated or
 * generated-by-generated; generated-by-reference (M_gr) is refused, since no score reads it. */
DUSTY_API int dusty_emd_matrix(const float* A, int na, int pa, const float* B, int nb, int pb,
                               int row_begin, int row_end, int row_stride, float* M, long long ldm,
                               int stacked_offset_a, int stacked_offset_b, int n_ref, int n_total, uint64_t* keys,
                               void* workspace, size_t workspace_bytes, void* stream);

/* --------------------------------------------------------------------------------------------
 * JSD between occupancy histograms (next row 8f-2; reference utils/metrics/jsd.py:23-121)
 * -------------------------------------------------------------------------------------------- */

/* Every point of pcs (b,npts,3) votes for its nearest in-sphere grid point (f32 arithmetic and
 * lowest-index tie rule of the reference's brute-force arg-min, jsd.py:59-69). The grid is supplied
 * by the caller exactly as the reference builds it (jsd.py:10-20): grid (ng,3) the in-sphere points
 * in order, cell_to_idx (res^3) their compact index or -1, axis (res) the coordinates along one axis.
 * counters (ng) u32: points per grid point (grid_counters); clouds_touching (ng) u32: number of
 * clouds with at least one point there (grid_bernoulli_rvars). Both are overwritten. */
DUSTY_API int dusty_jsd_vote(const float* pcs, int b, int npts, int resolution, int ng, const float* grid,
                             const int32_t* cell_to_idx, const float* axis, float spacing,
                             uint32_t* counters, uint32_t* clouds_touching, void* stream);

/* _jensen_shannon_divergence of two count vectors (jsd.py:110-121), base-2 entropies; out[0] f32. */
DUSTY_API int dusty_jsd_from_counts(const uint32_t* counts_p, const uint32_t* counts_q, int ng, float* out,
                                    void* stream);

/* --------------------------------------------------------------------------------------------
 * Farthest-point sampling
 * -------------------------------------------------------------------------------------------- */

DUSTY_API size_t dusty_fps_workspace_bytes(int b, int n, int m);

/* Iterative farthest-point sampling of m indices per cloud, bit-identical to the reference kernel:
 *   idx[i,0] = 0; a point takes part iff (double)fma(z,z,fma(x,x,y*y)) > 1e-3; running distances
 *   start at 1e10 and are evaluated as fma(dz,dz,fma(dx,dx,dy*dy)); among equal maxima the winner
 *   minimises (bitreverse_{log2 T}(k mod T), k div T) with T = min(2^floor(log2 n), 512), the
 *   outcome of the reference's strided scan + shared-memory tree.
 *   xyz (b,n,3) f32 contiguous; idx (b,m) i32; out_xyz (b,m,3) f32 gathered points or NULL. */
DUSTY_API int dusty_fps(const float* xyz, int b, int n, int m, int32_t* idx, float* out_xyz,
              void* workspace, size_t workspace_bytes, void* stream);

/* out[i,c,j] = points[i,c,idx[i,j]];  points (b,c,n), idx (b,m), out (b,c,m). */
DUSTY_API int dusty_gather_points(const float* points, const int32_t* idx, int b, int c, int n, int m,
                        float* out, void* stream);
/* grad_points (b,c,n) = scatter-add of grad_out (b,c,m) through idx; overwritten. */
DUSTY_API int dusty_gather_points_grad(const float* grad_out, const int32_t* idx, int b, int c, int n, int m,
                             float* grad_points, void* stream);

/* --------------------------------------------------------------------------------------------
 * Point-drop head + inverse spherical projection
 * -------------------------------------------------------------------------------------------- */

/* l = -log(log(u1 + eps) / log(u2 + eps) + eps), element-wise over count values. */
DUSTY_API int dusty_logistic_noise(const float* u1, const float* u2, float eps, size_t count, float* out,
                         void* stream);

/* One Gumbel-sigmoid gate (GumbelSigmoid, models/dusty.py:6-62): how its relaxed-Bernoulli noise is supplied, and
 * the gate's own scalars. DUSty-II has two gates, and each keeps its own temperature, eps and output kind. */
#define DUSTY_NOISE_NONE     0   /* gate is (logit > 0), DUSty2's eval-mode image gate */
#define DUSTY_NOISE_LOGISTIC 1   /* noise_a holds l */
#define DUSTY_NOISE_UNIFORM  2   /* noise_a, noise_b hold U1, U2; l as dusty_logistic_noise forms it, with the gate's eps */

typedef struct dusty_gate {
  int32_t mode;             /* DUSTY_NOISE_* */
  int32_t hard;             /* 1: straight-through (hard - soft) + soft, hard = soft > threshold; 0: the soft mask
                               (GumbelSigmoid(hard=False), models/dusty.py:58-59) */
  const float* noise_a;     /* l or U1 */
  const float* noise_b;     /* U2 or NULL */
  int64_t batch_stride;     /* elements between images in noise_a/b; 0 = one map shared by the batch */
  int64_t pixel_stride;     /* 1 = per-pixel map; 0 = one value per image */
  float inv_tau;            /* f32(1.0/tau): ATen CUDA forms x/scalar as x * f32(1/double(scalar)); for the learnable
                               temperature (tau=None, models/dusty.py:39-41) the f32 value of softplus(weight) + 1/tau_max */
  float eps;                /* 1e-10; used when mode == DUSTY_NOISE_UNIFORM */
} dusty_gate;

typedef struct dusty_head_params {
  int32_t b, h, w;
  int32_t conf_channels;    /* 1 (DUSty-I) or 2 (DUSty-II: channel 0 pixel gate, channel 1 image gate) */
  dusty_gate gate_pixel;
  dusty_gate gate_image;    /* ignored when conf_channels == 1 */
  float threshold;          /* mask_soft > threshold, the same for both gates as in the reference */
  float drop_const;         /* generator-side drop value, -1 */
  /* projection constants, exactly the f32 scalars the reference's element-wise kernels receive */
  float tol;                /* |inv - 0| > tol */
  float disp_scale;         /* f32(1/min_depth - 1/max_depth) */
  float disp_shift;         /* f32(1/max_depth) */
  float min_depth;          /* f32(min_depth) */
  float inv_range;          /* f32(1.0 / (max_depth - min_depth)), reciprocal in double */
  float range;              /* f32(max_depth - min_depth) */
  float inv_max_depth;      /* f32(1.0 / max_depth) */
  int32_t points_layout;    /* 0: xyz planar (b,3,h,w) like inv_to_xyz; 1: interleaved (b,h*w,3) */
} dusty_head_params;

/* GumbelSigmoid.forward alone (models/dusty.py:45-59): soft = 1/(1+exp(-((logit + l) * gate->inv_tau))); out is
 * (hard - soft) + soft with hard = soft > threshold when gate->hard, else soft. A NaN threshold is an ordinary
 * threshold: no soft value exceeds it, so a hard gate returns exact zeros, as the reference does.
 * logits/out (b,1,h*w) f32, 16-byte aligned, npix a multiple of 4. */
DUSTY_API int dusty_gumbel_sigmoid(const float* logits, const dusty_gate* gate, float threshold, int b, int npix,
                         float* out, void* stream);

/* Fused point-drop head + projection.
 *   depth (b,1,h,w), confidence (b,C,h,w): generator outputs (tanh range).
 *   trig (4,h,w): cos(elev), sin(elev), cos(azim), sin(azim) of the LiDAR angle grid; may be NULL
 *   when neither out_points nor compaction is requested (maskout alone).
 *   out_mask (b,C,h,w), out_depth (b,1,h,w): DUSty{1,2}.maskout results; out_points: xyz.
 *   Optional compaction (all three NULL to disable): out_count (b) i32 = number of valid pixels
 *   (inv != 0 within tol), out_index (b,h*w) i32 = their pixel indices in ascending order,
 *   out_compact (b,h*w,3) f32 = their xyz in that order; tails are left untouched.
 *   All tensor pointers must be 16-byte aligned and w a multiple of 4. */
DUSTY_API size_t dusty_head_project_workspace_bytes(int b, int h, int w);
DUSTY_API int dusty_head_project(const dusty_head_params* p, const float* depth, const float* confidence,
                       const float* trig, float* out_mask, float* out_depth, float* out_points,
                       int32_t* out_count, int32_t* out_index, float* out_compact,
                       void* workspace, size_t workspace_bytes, void* stream);

/* Backward of dusty_head_project: the gradient autograd gives through the reference's op chain (GumbelSigmoid's
 * straight-through estimator, the mask blend, tanh_to_sigmoid + clamp, inv_to_xyz), with every forward value
 * recomputed bit-identically from the forward's inputs; nothing is saved by the forward.
 *   p, depth, confidence: exactly what the forward received, gate noise pointers included.
 *   Upstream gradients, each NULL for zero: grad_mask (b,C,h,w), grad_depth (b,1,h,w), grad_points in
 *   p->points_layout. trig (4,h,w) is required when grad_points is given.
 *   grad_depth_in (b,1,h,w), grad_confidence (b,C,h,w): overwritten. Channel 1 of a DUSty-II gate without noise
 *   (DUSTY_NOISE_NONE, eval mode) is 0.
 *   grad_inv_tau: NULL, or conf_channels floats: d loss / d gate_pixel.inv_tau, then (DUSty-II) d loss /
 *   d gate_image.inv_tau; 0 for a gate without noise. It needs dusty_head_project_backward_workspace_bytes() of
 *   workspace, and each float is reduced in a fixed order (no atomics), so repeated calls give bit-identical results.
 *   All tensor pointers must be 16-byte aligned and w a multiple of 4. */
DUSTY_API size_t dusty_head_project_backward_workspace_bytes(int b, int h, int w);
DUSTY_API int dusty_head_project_backward(const dusty_head_params* p, const float* depth, const float* confidence,
                       const float* trig, const float* grad_mask, const float* grad_depth, const float* grad_points,
                       float* grad_depth_in, float* grad_confidence, float* grad_inv_tau,
                       void* workspace, size_t workspace_bytes, void* stream);

/* Projection only: inv (b,1,h,w) in [0,1] (already tanh_to_sigmoid'ed and clamped) -> xyz. */
DUSTY_API int dusty_inv_to_xyz(const dusty_head_params* p, const float* inv, const float* trig,
                     float* out_points, void* stream);

/* --------------------------------------------------------------------------------------------
 * Real-data side: organised LiDAR scans -> range images + clouds (the reference set of the evaluation)
 * -------------------------------------------------------------------------------------------- */

typedef struct dusty_scan_params {
  int32_t b, hs, ws;        /* scans (b,hs,ws,channels) f32 as process_kitti.py stores them: (64,2048,4) */
  int32_t channels;         /* >= 3; xyz are channels 0..2 (channel 3 = reflectance, unused on this path) */
  int32_t h, w;             /* output range-image shape; w a multiple of 4 */
  float scale_h, scale_w;   /* f32(hs)/h, f32(ws)/w: source index = min((int)floorf(dst*scale), size-1),
                               torch's nearest interpolation (torchvision TF.resize(..., NEAREST)) */
  float min_depth;          /* f32(min_depth): mask = r > 0 && r > min_depth && r < max_depth */
  float max_depth;          /* f32(max_depth); also xyz /= max_depth (true division) */
  float range;              /* f32(max_depth - min_depth): depth = (r - min_depth) / range (true division) */
  /* invert_depth + sigmoid_to_tanh as ATen's CUDA element-wise kernels round them */
  float disp_lo;            /* f32(1/max_depth) */
  float inv_disp_range;     /* f32(1.0 / (1/min_depth - 1/max_depth)) */
  float drop_const;         /* generator-side drop value (-1): inv = mask*inv + (1-mask)*drop_const */
} dusty_scan_params;

/* One pass over a batch of scans. Outputs (any of out_depth / out_xyz may be NULL):
 *   out_depth  (b,1,h,w)  normalised range in [0,1], 0 where masked        (dataset "depth")
 *   out_mask   (b,1,h,w)  1.0 / 0.0                                         (dataset "mask", .float())
 *   out_inv    (b,1,h,w)  tanh-space inverse depth, drop_const where masked (preprocess_reals "inv")
 *   out_points (b,h*w,3)  unit-space xyz, interleaved (what FPS consumes); origin where masked
 *   out_xyz    (b,3,h,w)  the same, planar                                  (dataset "xyz")
 * scans must be 4-byte aligned (16-byte when channels == 4 for the vector path, checked at run
 * time); outputs 16-byte aligned. */
DUSTY_API int dusty_scan_preprocess(const dusty_scan_params* p, const float* scans, float* out_depth,
                          float* out_mask, float* out_inv, float* out_points, float* out_xyz, void* stream);

/* --------------------------------------------------------------------------------------------
 * Measurement helper (bench.py only): sustained dependent-free FFMA rate, for the FP32 roofline.
 * Runs `iters` rounds of 4096 FFMA per thread on a full grid; writes elapsed device milliseconds.
 * -------------------------------------------------------------------------------------------- */
DUSTY_API int dusty_probe_fp32_peak(int iters, float* sink, double* flops_out, void* stream);

/* Measurement helper (bench.py only): the merged-origin / pruned Chamfer kernels skip candidate chunks by an exact
 * box bound, so the number of (row, candidate) pairs they evaluate is data dependent. enable != 0 switches a device
 * counter on (per process and current device; the kernels then add to it with one atomic per warp and tile),
 * enable == 0 switches it off; either way *pairs_out (may be NULL) receives the count accumulated since the last
 * call and the counter restarts at zero. Not for timed runs: the call synchronises the device. */
DUSTY_API int dusty_chamfer_count_pairs(int enable, uint64_t* pairs_out);

#ifdef __cplusplus
}
#endif
#endif /* DUSTY_B200_H_ */
