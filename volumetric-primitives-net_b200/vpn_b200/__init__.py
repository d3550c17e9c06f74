"""vpn_b200 - B200-native (sm_100a) primitive assembly + loss hot path of Volumetric-Primitives-Net.

Host-side mirror of the reference's Python call surface over libvpn_b200.so (include/vpn_b200.h).
"""
from .ops import (CHAMFER_AUTO, CHAMFER_GENERIC, CHAMFER_TILED_EXACT, CHAMFER_TILED_FMA, CHAMFER_TILED_EXPAND, CHAMFER_TILED_TC,
                  chamfer_distance, chamfer_main_kernel_name, chamfer_nn, chamfer_nn_stage_ms, cuboid_face_counts, emd_auction, emd_distance, fp32_peak_tflops, image_bounds, look_at_cameras, mesh_vertices, mesh_vertices_mixed, perceptual_feature_pooling,
                  obj_to_view_points, sample_mesh_surface, sample_mixed_primitives, sample_primitives, sample_primitives_ms, soft_silhouette, transform_points, view_to_obj_points)
from .step import GraphedMeshLoss, GraphedPrimitiveLoss, HostPipeline, MeshLoss, MeshLossConfig, PrimitiveLoss, PrimitiveLossConfig
from ._lib import VpnError, LIB_PATH

__all__ = [
    "CHAMFER_AUTO", "CHAMFER_GENERIC", "CHAMFER_TILED_EXACT", "CHAMFER_TILED_FMA", "CHAMFER_TILED_EXPAND", "CHAMFER_TILED_TC", "chamfer_distance", "chamfer_main_kernel_name", "chamfer_nn", "chamfer_nn_stage_ms",
    "cuboid_face_counts", "emd_auction", "emd_distance", "image_bounds", "perceptual_feature_pooling", "fp32_peak_tflops", "look_at_cameras", "mesh_vertices", "mesh_vertices_mixed", "obj_to_view_points",
    "sample_mesh_surface", "sample_mixed_primitives", "sample_primitives", "sample_primitives_ms", "soft_silhouette", "transform_points", "view_to_obj_points", "GraphedMeshLoss", "GraphedPrimitiveLoss", "HostPipeline", "MeshLoss", "MeshLossConfig", "PrimitiveLoss",
    "PrimitiveLossConfig", "VpnError", "LIB_PATH",
]
