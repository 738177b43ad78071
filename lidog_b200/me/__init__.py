"""Host-side mirror of the MinkowskiEngine 0.5.4 surface LiDOG uses (SURVEY.md section 2.2),
backed by liblidog_b200 (sm_100a).  Import as `import MinkowskiEngine as ME` through the
top-level alias package, or as `from lidog_b200 import me as ME`."""
from .sparse_tensor import SparseTensor, CoordinateMapKey, cat
from .coords import CoordinateManager
from .conv import MinkowskiConvolution, MinkowskiConvolutionTranspose, MinkowskiConvolutionBase, SparseConvFunction
from .norm import (MinkowskiBatchNorm, MinkowskiSyncBatchNorm, MinkowskiInstanceNorm, MinkowskiReLU,
                   MinkowskiDropout)
from .isw import instance_covariance, instance_whitening_loss
from . import utils, modules

__version__ = "0.5.4+lidog_b200"
