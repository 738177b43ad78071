"""Drop-in `MinkowskiEngine` package name for LiDOG: re-exports lidog_b200.me.
Put the repository root on PYTHONPATH and the reference's `import MinkowskiEngine as ME`
(train_lidog.py:11, utils/models/minkunet_bev.py:2, utils/collation/collation.py:2) resolves here."""
from lidog_b200.me import *  # noqa: F401,F403
from lidog_b200.me import (SparseTensor, CoordinateMapKey, cat, CoordinateManager, MinkowskiConvolution,
                           MinkowskiConvolutionTranspose, MinkowskiBatchNorm, MinkowskiSyncBatchNorm,
                           MinkowskiInstanceNorm, MinkowskiReLU, MinkowskiDropout, __version__)
from . import utils, modules  # noqa: F401
