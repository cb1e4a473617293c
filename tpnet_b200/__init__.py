"""tpnet_b200 — B200 (sm_100a) implementation of TPNet's temporal-walk-matrix
projection hot path (reference: models/TPNet.py:9-157 of lxd99/TPNet).

    from tpnet_b200 import RandomProjectionModule      # drop-in for models.TPNet.RandomProjectionModule
"""
from .negative_sampler import NegativeEdgeSampler  # noqa: F401
from .random_projection import RandomProjectionModule  # noqa: F401

__all__ = ['NegativeEdgeSampler', 'RandomProjectionModule']
