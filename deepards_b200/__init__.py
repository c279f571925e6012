"""deepards_b200 -- B200 (sm_100a) backend for the deepards cnn_linear hot path.

Public surface = the reference's plugin surface for this path:
  * backbone factories    resnet18 / 34 / 50 / 101 / 152, densenet18 / densenet121   (deepards/models/resnet.py, densenet.py)
  * heads                 CNNLinearNetwork / CNNSingleBreathLinearNetwork  (deepards/models/torch_cnn_linear_network.py)
  * registries            base_networks / network_heads, install()         (deepards/train_ards_detector.py:45-69, 1410-1436)
plus the data-parallel trainer (data_parallel.DataParallelTrainer) that replaces nn.DataParallel
(train_ards_detector.py:93-96).
"""
from .resnet import resnet18, resnet34, resnet50, resnet101, resnet152, ResNet, BasicBlock, Bottleneck  # noqa: F401
from .densenet import densenet18, densenet121, DenseNet  # noqa: F401
from .torch_cnn_linear_network import (CNNLinearNetwork, CNNSingleBreathLinearNetwork, CNNLinearToMean,  # noqa: F401
                                       CNNLinearComprToRF, CNNDoubleLinearNetwork, CNNRegressor, CNNLSTMNetwork,
                                       CNNTransformerNetwork)
from .input_pipeline import WindowScaler  # noqa: F401
from . import gradcam  # noqa: F401
from .patient_votes import patient_vote_table  # noqa: F401
from .registry import base_networks, network_heads, install  # noqa: F401

__all__ = ["resnet18", "resnet34", "resnet50", "resnet101", "resnet152", "densenet18", "densenet121", "ResNet", "DenseNet",
           "BasicBlock", "Bottleneck", "CNNLinearNetwork",
           "CNNSingleBreathLinearNetwork", "CNNLinearToMean", "CNNLinearComprToRF", "CNNDoubleLinearNetwork",
           "CNNRegressor", "CNNLSTMNetwork", "CNNTransformerNetwork", "patient_vote_table", "WindowScaler", "gradcam", "base_networks", "network_heads", "install"]
