"""myria3d_b200 -- B200-native (sm_100a) RandLA-Net hot path for IGNF/myria3d.

Host side: Python / PyTorch (device memory, streams, autograd plumbing).
Device side: ``libb200randla.so`` -- hand-written CUDA behind the C ABI of ``include/b200randla.h``.
"""
from .randla_net import B200Block1Net, B200RandLANet  # noqa: F401
from .model import MODEL_ZOO, Model, get_neural_net_class  # noqa: F401
from .data import Batch, Data  # noqa: F401
from .batch_prep import PrepConfig, RawCollater, prepare_batch  # noqa: F401

__version__ = "0.1.0"
