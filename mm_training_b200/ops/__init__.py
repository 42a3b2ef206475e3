# operator packages mirror the reference's ``ops/`` layout: ``from mm_training_b200.ops.voxel_pooling import voxel_pooling``
from .bev_augment import warp_affine

__all__ = ['warp_affine']
