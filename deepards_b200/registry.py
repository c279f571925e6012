"""The reference's two plugin registries for this path, resolved to the B200 implementations.

`base_networks` (deepards/train_ards_detector.py:45-69) maps `--base-network` names to backbone factories;
`network_map` (:1410-1436) maps `--network` names to trainer classes whose `get_network(base_network)` builds the
head (:938-939, :963-964).  `install(module)` patches a loaded `train_ards_detector` module in place, so that
`train_ards_detector.py --network cnn_linear --base-network resnet18|densenet18` builds the networks of this
package with no other change (INTEGRATION.md shows the two-line edit a maintainer would make instead).
"""
from .densenet import densenet18, densenet121
from .resnet import resnet18, resnet34, resnet50, resnet101, resnet152
from .torch_cnn_linear_network import (CNNDoubleLinearNetwork, CNNLinearComprToRF, CNNLinearNetwork, CNNLinearToMean,
                                       CNNLSTMNetwork, CNNRegressor, CNNSingleBreathLinearNetwork, CNNTransformerNetwork)

base_networks = {
    'resnet18': resnet18,
    'resnet34': resnet34,
    'resnet50': resnet50,
    'resnet101': resnet101,
    'resnet152': resnet152,
    'densenet18': densenet18,
    'densenet121': densenet121,
}

# --network name -> head class built by the trainer's get_network()
network_heads = {
    'cnn_linear': CNNLinearNetwork,
    'cnn_single_breath_linear': CNNSingleBreathLinearNetwork,
    'cnn_linear_to_mean': CNNLinearToMean,
    'cnn_linear_compr_to_rf': CNNLinearComprToRF,
    'cnn_double_linear': CNNDoubleLinearNetwork,
    'cnn_regressor': CNNRegressor,
    'cnn_lstm': CNNLSTMNetwork,
    'cnn_transformer': CNNTransformerNetwork,
}


def install(train_module):
    """Patch `deepards.train_ards_detector` (already imported) to construct B200 networks."""
    train_module.base_networks.update(base_networks)
    train_module.CNNLinearNetwork = CNNLinearNetwork
    train_module.CNNSingleBreathLinearNetwork = CNNSingleBreathLinearNetwork
    for cls in (CNNLinearToMean, CNNLinearComprToRF, CNNDoubleLinearNetwork, CNNRegressor, CNNLSTMNetwork,
                CNNTransformerNetwork):
        setattr(train_module, cls.__name__, cls)
    return train_module
