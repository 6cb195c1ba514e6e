"""dusty-gan_b200: B200-native kernels behind DUSty-GAN's generate-and-evaluate hot path.

The package mirrors the reference's module paths for that path and nothing else:

    models.dusty                 GumbelSigmoid, DUSty1, DUSty2          (reference models/dusty.py)
    utils                        tanh_to_sigmoid, sigmoid_to_tanh, flatten (reference utils/__init__.py:70-79,213)
    utils.lidar                  Coordinate, LiDAR                      (reference utils/lidar.py)
    utils.sampling.fps           furthest_point_sampling, gather_operation, downsample_point_clouds
    utils.metrics.distance       chamfer_distance, ChamferDistance, earth_mover_distance
    utils.metrics.cov_mmd_1nna   compute_cd, compute_emd, emd_matrix, _pairwise_distance, compute_cov_mmd_1nna
    utils.metrics.jsd            compute_jsd                              (reference utils/metrics/jsd.py)
    datasets                     define_dataset, KITTIOdometry, preprocess_scans (reference datasets/kitti.py)
    pipeline                     fused generate->points entry (project_2d_to_3d of evaluate_synthesis.py:59-64),
                                 preprocess_reals / build_real_cache (evaluate_synthesis.py:49-57, 69-110)
    sharding                     row-sharded Chamfer matrix over torch.distributed

All compute goes through ``libdustyb200.so`` (C ABI in include/dusty_b200.h); there is no CPU or
PyTorch fallback: calling an op without the library or without a CUDA tensor raises.
"""
__version__ = "0.1.0"
