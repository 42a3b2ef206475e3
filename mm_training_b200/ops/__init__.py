# operator packages mirror the reference's ``ops/`` layout: ``from mm_training_b200.ops.voxel_pooling import voxel_pooling``
from .bev_augment import warp_affine
from .depth_loss import depth_loss

__all__ = ['warp_affine', 'depth_loss']
