"""haf_grasping_b200 -- B200-native (sm_100a) grasp-search hot path of haf_grasping behind a C ABI.

Layout: csrc/ (CUDA kernels + the C ABI, built into lib/libhafgpu.so), api.py (ctypes binding),
pcd.py (PCD ingest), synth.py (synthetic workloads).  No CPU fallback exists.
"""
from .api import (GraspSearch, HafError, SvmPredictor, scale_apply, scale_minmax, build_transform, haf_best, haf_candidate, haf_depth_image, haf_grasp, haf_rank_params, haf_request, load_library, make_request, make_requests,  # noqa: F401
                  HAF_DEPTH_F32, HAF_DEPTH_U16, HAF_SVM_FP32_GUARD, HAF_SVM_FP64_EXACT, HAF_SVM_TENSOR_GUARD)
