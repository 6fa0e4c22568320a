"""dirt_b200 -- a B200-native (sm_100a) differentiable rasteriser behind the dirt.rasterise API.

`import dirt_b200 as dirt` is the drop-in for the reference package (dirt/__init__.py:1-3).
"""
from .rasterise_ops import rasterise, rasterise_batch, rasterise_batch_shared, rasterise_deferred, rasterise_batch_deferred
from . import matrices, lighting, projection

__all__ = ['rasterise', 'rasterise_batch', 'rasterise_batch_shared', 'rasterise_deferred', 'rasterise_batch_deferred',
           'matrices', 'lighting', 'projection']
