"""mc3_b200 -- B200-native (sm_100a) implementation of the sampling hot path of
pcubillos/mc3 behind mc3's own API.

    import mc3_b200 as mc3
    out = mc3.sample(data, uncert, func=mc3.models.sinusoid, params=..., indparams=[x],
                     sampler='demc', nchains=4096, nsamples=4e6, ...)

Host code is Python (torch tensors for device memory, streams, graphs and
torch.distributed); the arithmetic is hand-written CUDA in libmc3b200.so, bound
through a C ABI (include/mc3b200.h) with ctypes.  There is no CPU fallback.
"""
from . import models
from .models import BuiltinModel, CudaModel, TorchModel
from .sampler_driver import sample, __version__
from .batch_driver import sample_batch
from .fit_driver import fit
from . import stats
from . import utils
from .utils import Log

__all__ = ['sample', 'sample_batch', 'fit', 'stats', 'utils', 'models', 'BuiltinModel',
           'CudaModel', 'TorchModel', 'Log', '__version__']
