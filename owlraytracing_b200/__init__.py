"""owlraytracing_b200 — B200-native TrueKNN hot path (LBVH build + warp-cooperative traversal).

Only what the path needs: `csrc/` (CUDA kernels + the C ABI of include/trueknn.h), the ctypes
loader, the host-side mirror of the sample's interface, the synthetic clouds of BASELINE.json and
the two multi-GPU drivers.  Importing the package does not require a GPU; creating a `TrueKNN`
does (there is no CPU fallback).
"""
from .trueknn import MultiTrueKNN, TrueKNN, TrueKNNError, batch_to_offsets, chamfer_distance, estimate_pointcloud_local_coord_frames, estimate_pointcloud_normals, feature_knn, feature_knn_graph, fps, grid_cluster, grid_sampling, knn, knn_graph, knn_interpolate, knn_points, radius, radius_graph, read_points, read_points_fast, run_sample, voxel_grid, write_neighbour_lists, write_neighbours  # noqa: F401
from . import datasets  # noqa: F401

__all__ = ["TrueKNN", "MultiTrueKNN", "TrueKNNError", "feature_knn", "feature_knn_graph", "fps", "grid_cluster", "voxel_grid", "grid_sampling", "knn", "knn_interpolate", "knn_points", "chamfer_distance", "estimate_pointcloud_normals", "estimate_pointcloud_local_coord_frames", "radius", "knn_graph", "radius_graph", "batch_to_offsets", "read_points", "read_points_fast", "write_neighbours", "write_neighbour_lists", "run_sample", "datasets"]
